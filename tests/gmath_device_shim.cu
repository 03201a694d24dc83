/* Device-side export of gmath.h for tests/test_gmath_device.py: the entry points of tests/gmath_host_shim.c under the
 * same names, each one kernel over the inputs.  An entry point copies its inputs to the device, runs the kernel,
 * copies the outputs back, frees what it allocated and returns the first CUDA error.  Built with the library's own
 * nvcc flags (gelato_b200/engine.py: NVCC_FLAGS), so the functions compile as they do in the kernels. */
#include <cuda_runtime.h>

#include "gmath_shim.h"

typedef void (*GmsKernel)(const double*, const double*, const double*, double*, double*, int);

/* nin inputs (a, b, c) and nout outputs (y, z) of n doubles each, through one device allocation */
static cudaError_t gms_run(GmsKernel k, int n, int nin, const double* a, const double* b, const double* c, int nout,
                           double* y, double* z) {
  if (n <= 0) return cudaSuccess;
  const size_t bytes = (size_t)n * sizeof(double);
  double* buf = nullptr;
  cudaError_t err = cudaMalloc(&buf, (size_t)(nin + nout) * bytes);
  if (err != cudaSuccess) return err;
  const double* in[3] = {a, b, c};
  double* out[2] = {y, z};
  double* d[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  for (int i = 0; i < nin + nout; i++) d[i] = buf + (size_t)i * n;
  for (int i = 0; i < nin && err == cudaSuccess; i++) err = cudaMemcpy(d[i], in[i], bytes, cudaMemcpyHostToDevice);
  if (err == cudaSuccess) {
    const int threads = 256;
    k<<<(n + threads - 1) / threads, threads>>>(d[0], nin > 1 ? d[1] : nullptr, nin > 2 ? d[2] : nullptr, d[nin],
                                                nout > 1 ? d[nin + 1] : nullptr, n);
    err = cudaGetLastError();
  }
  for (int i = 0; i < nout && err == cudaSuccess; i++) err = cudaMemcpy(out[i], d[nin + i], bytes, cudaMemcpyDeviceToHost);
  const cudaError_t ferr = cudaFree(buf);
  return err != cudaSuccess ? err : ferr;
}

#define GMS_KERNEL_HEAD(name)                                                                                        \
  __global__ void gmk_##name(const double* pa, const double* pb, const double* pc, double* py, double* pz, int n) { \
    const int i = blockIdx.x * blockDim.x + threadIdx.x;                                                            \
    if (i >= n) return;

#define U(name, expr)                                                                                     \
  GMS_KERNEL_HEAD(name)                                                                                   \
  const double a = pa[i];                                                                                 \
  py[i] = expr;                                                                                           \
  }                                                                                                       \
  extern "C" cudaError_t gmt_##name(const double* x, double* y, int n) {                                  \
    return gms_run(gmk_##name, n, 1, x, nullptr, nullptr, 1, y, nullptr);                                 \
  }
#define B(name, expr)                                                                                     \
  GMS_KERNEL_HEAD(name)                                                                                   \
  const double a = pa[i], b = pb[i];                                                                      \
  py[i] = expr;                                                                                           \
  }                                                                                                       \
  extern "C" cudaError_t gmt_##name(const double* x, const double* w, double* y, int n) {                 \
    return gms_run(gmk_##name, n, 2, x, w, nullptr, 1, y, nullptr);                                       \
  }
#define T(name, expr)                                                                                     \
  GMS_KERNEL_HEAD(name)                                                                                   \
  const double a = pa[i], b = pb[i], c = pc[i];                                                           \
  py[i] = expr;                                                                                           \
  }                                                                                                       \
  extern "C" cudaError_t gmt_##name(const double* x, const double* w, const double* v, double* y, int n) { \
    return gms_run(gmk_##name, n, 3, x, w, v, 1, y, nullptr);                                             \
  }
#define U2(name, stmt)                                                                                    \
  GMS_KERNEL_HEAD(name)                                                                                   \
  const double a = pa[i];                                                                                 \
  double y0, y1;                                                                                          \
  stmt;                                                                                                   \
  py[i] = y0;                                                                                             \
  pz[i] = y1;                                                                                             \
  }                                                                                                       \
  extern "C" cudaError_t gmt_##name(const double* x, double* y, double* z, int n) {                       \
    return gms_run(gmk_##name, n, 1, x, nullptr, nullptr, 2, y, z);                                       \
  }
GMATH_SHIM_ENTRIES(U, B, T, U2)
