// Move-only owners of the CUDA resources a plan holds: device and page-locked host arrays, streams, events and a
// graph exec.  Each releases what it owns when it is destroyed, so a plan frees everything by being deleted.
// Host code only.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <utility>

namespace gelato_host {

// An array of T in device memory (Pinned = false) or page-locked host memory (Pinned = true).
template <typename T, bool Pinned>
class Buffer {
 public:
  Buffer() = default;
  Buffer(Buffer&& o) noexcept : ptr_(std::exchange(o.ptr_, nullptr)), size_(std::exchange(o.size_, 0)) {}
  ~Buffer() { release(); }

  // Room for n elements.  Nothing happens when there is room already; otherwise the old storage is freed before the
  // new one is allocated (its contents are lost).  cudaFree synchronises the device: no launch still uses the old
  // storage once this returns.
  cudaError_t reserve(size_t n) {
    if (n <= size_) return cudaSuccess;
    release();
    void* p = nullptr;
    const cudaError_t e = Pinned ? cudaMallocHost(&p, n * sizeof(T)) : cudaMalloc(&p, n * sizeof(T));
    if (e != cudaSuccess) return e;
    ptr_ = static_cast<T*>(p);
    size_ = n;
    return cudaSuccess;
  }

  T* get() const { return ptr_; }
  size_t size() const { return size_; }

 private:
  void release() {
    if (ptr_ && Pinned) cudaFreeHost(ptr_);
    if (ptr_ && !Pinned) cudaFree(ptr_);
    ptr_ = nullptr;
    size_ = 0;
  }
  T* ptr_ = nullptr;
  size_t size_ = 0;
};

template <typename T>
using DeviceBuf = Buffer<T, false>;
template <typename T>
using PinnedBuf = Buffer<T, true>;

// A CUDA handle (stream, event, graph exec) and the call that destroys it.
template <typename H, cudaError_t (*Destroy)(H)>
class Handle {
 public:
  Handle() = default;
  explicit Handle(H h) : h_(h) {}
  Handle(Handle&& o) noexcept : h_(std::exchange(o.h_, nullptr)) {}
  Handle& operator=(Handle&& o) noexcept {
    std::swap(h_, o.h_);
    return *this;
  }
  ~Handle() { reset(); }

  operator H() const { return h_; }
  void reset() {
    if (h_) Destroy(h_);
    h_ = nullptr;
  }
  // where a create call writes the new handle; whatever was owned before is destroyed first
  H* out() {
    reset();
    return &h_;
  }

 private:
  H h_ = nullptr;
};

using Stream = Handle<cudaStream_t, cudaStreamDestroy>;
using Event = Handle<cudaEvent_t, cudaEventDestroy>;
using GraphExec = Handle<cudaGraphExec_t, cudaGraphExecDestroy>;

}  // namespace gelato_host
