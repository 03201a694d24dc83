// gelato_b200.cu -- CUDA kernels (sm_100a) and the C ABI declared in
// include/gelato_b200.h.
//
// Two fused kernels cover the whole NLP callback path:
//   k_residuals : everything `objfunc` evaluates (Trajectory_Optimization.py:194-242)
//   k_jacobian  : every x-dependent Jacobian value `sens` produces (:245-312)
// Each is ONE launch per call; blocks take their role from a block table built
// at plan creation (dynamics sections in chunks of nodes, aero rows, event
// rows, linear rows), one copy of the block list per scenario of a batched solve.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false (see DESIGN.md H1;
// gelato_selftest_unfused() verifies the flag at run time).
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "cuda_owned.h"
#include "host_pool.h"
#include "mesh_error.h"
#include "plan_host.h"
#include "user_table.h"

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
// One Jacobian evaluation = ONE launch: every role's blocks, heavy (air dynamics nodes, aero rows: the pos_part /
// rotq_part code, ~1 kFLOP per column) and light (vacuum dynamics, fallback, event rows) interleaved in the block
// table so that FP64-issue-bound and latency-bound blocks share each SM.  (Round 2 first split the roles into two
// kernels on two streams: they ran one after the other -- the first kernel fills every SM -- and the instruction
// cache hit rate did not move; profiles/r02a_ab_probe.txt.)  The role-subset instantiations below exist for
// measurements only (gelato_launch_kernel_dev).
#ifndef GJ_MIN_BLOCKS
#define GJ_MIN_BLOCKS 2 /* 448 threads x 2 blocks: 28 warps per SM, up to 72 registers */
#endif
// The blocks of the first wave ask L2 for the whole decision-vector batch (one 128-byte line per thread, no
// register, no wait): a block reads ~25 scattered lines of x before it can start, and on an L2 that does not hold
// them every later wave would pay the DRAM latency again.  0 switches it off.
#ifndef GJ_PREFETCH_BLOCKS
#define GJ_PREFETCH_BLOCKS 296
#endif
__device__ __forceinline__ void prefetch_batch_l2(const double* x_all, size_t n_doubles, int blocks, int threads) {
#if GJ_PREFETCH_BLOCKS > 0
  if ((int)blockIdx.x < blocks) {
    const size_t lines = (n_doubles * sizeof(double) + 127) / 128;
    for (size_t l = (size_t)blockIdx.x * threads + threadIdx.x; l < lines; l += (size_t)blocks * threads)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(x_all) + l * 128));
  }
#endif
}
// Measurement build only (-DGJ_CLOCKS): cycles every warp spends in each phase and at each barrier, summed per
// (role, warp) over the launch; read back with gelato_debug_clocks (tools/phase_clocks.py).
#ifdef GJ_CLOCKS
__device__ unsigned long long gj_clk_sum[8][16][6];  // [role][warp][phase0, wait0, phase2, wait2, phase3, blocks]
#define GJ_CLK_DECL long long clk_[6] = {0, 0, 0, 0, 0, 0}
#define GJ_CLK(i) clk_[i] = clock64()
#define GJ_CLK_FLUSH(role, two)                                                                         \
  if ((threadIdx.x & 31) == 0) {                                                                        \
    unsigned long long* c = gj_clk_sum[(role) & 7][threadIdx.x >> 5];                                   \
    atomicAdd(c + 0, (unsigned long long)(clk_[1] - clk_[0]));                                              \
    atomicAdd(c + 1, (unsigned long long)(clk_[2] - clk_[1]));                                              \
    atomicAdd(c + 2, (unsigned long long)((two) ? 0 : clk_[3] - clk_[2]));                                  \
    atomicAdd(c + 3, (unsigned long long)((two) ? 0 : clk_[4] - clk_[3]));                                  \
    atomicAdd(c + 4, (unsigned long long)(clk_[5] - clk_[4]));                                              \
    atomicAdd(c + 5, 1ull);                                                                             \
  }
#else
#define GJ_CLK_DECL
#define GJ_CLK(i)
#define GJ_CLK_FLUSH(role, two)
#endif
template <int ROLES>
__device__ __forceinline__ void jacobian_body(const PlanView& P, const int32_t* __restrict__ block_table, const int n_scen,
                                              const int32_t* __restrict__ scen_ids, const double* __restrict__ x_all,
                                              double* __restrict__ out_all, double* __restrict__ g_all) {
  __shared__ JacStore store;
  const JacScratch sm = jac_scratch(store);
  prefetch_batch_l2(x_all, (size_t)n_scen * P.n_vars, GJ_PREFETCH_BLOCKS, GJ_THREADS);
  // block-major launch order: block b of every scenario before block b+1 of any
  const int scen = blockIdx.x % n_scen;
  const int32_t* bt = block_table + (size_t)(blockIdx.x / n_scen) * BT_COLS;
  const double* x = x_all + (size_t)scen * P.n_vars;
  // COO output: vals[n_scen][n_vals] (constants pre-filled); packed output: [n_scen][n_pack]
  double* out = out_all + (size_t)scen * (size_t)(P.packed ? P.n_pack : P.n_vals);
  // pair evaluation: every block also writes objfunc's rows of its nodes / constraint rows / events
  double* g = g_all ? g_all + (size_t)scen * P.n_rows : nullptr;
  // which scenario's parameter blocks this batch slot uses (a coalesced subset of the configured scenarios)
  const int sid = scen_ids ? scen_ids[scen] : scen;
  const bool two_phase = jac_role_two_phase(bt[BT_ROLE]);
  GJ_CLK_DECL;
  GJ_CLK(0);
  jac_block_phase<ROLES>(P, sid, bt, x, out, g, threadIdx.x, 0, sm);
  GJ_CLK(1);
  __syncthreads();
  GJ_CLK(2);
  if (!two_phase) {
    jac_block_phase<ROLES>(P, sid, bt, x, out, g, threadIdx.x, 2, sm);
    GJ_CLK(3);
    __syncthreads();
  }
  GJ_CLK(4);
  jac_block_phase<ROLES>(P, sid, bt, x, out, g, threadIdx.x, 3, sm);
  GJ_CLK(5);
  GJ_CLK_FLUSH(bt[BT_ROLE], two_phase);
}
__global__ void __launch_bounds__(GJ_THREADS, GJ_MIN_BLOCKS)
k_jacobian(const __grid_constant__ PlanView P, const int32_t* __restrict__ block_table, const int n_scen, const int32_t* __restrict__ scen_ids,
           const double* __restrict__ x_all, double* __restrict__ out_all, double* __restrict__ g_all) {
  jacobian_body<JR_ALL>(P, block_table, n_scen, scen_ids, x_all, out_all, g_all);
}
__global__ void __launch_bounds__(GJ_THREADS, GJ_MIN_BLOCKS)
k_jacobian_heavy(const __grid_constant__ PlanView P, const int32_t* __restrict__ block_table, const int n_scen,
                 const int32_t* __restrict__ scen_ids, const double* __restrict__ x_all, double* __restrict__ out_all,
                 double* __restrict__ g_all) {
  jacobian_body<JR_HEAVY>(P, block_table, n_scen, scen_ids, x_all, out_all, g_all);
}
__global__ void __launch_bounds__(GJ_THREADS, GJ_MIN_BLOCKS)
k_jacobian_light(const __grid_constant__ PlanView P, const int32_t* __restrict__ block_table, const int n_scen,
                 const int32_t* __restrict__ scen_ids, const double* __restrict__ x_all, double* __restrict__ out_all,
                 double* __restrict__ g_all) {
  jacobian_body<JR_LIGHT>(P, block_table, n_scen, scen_ids, x_all, out_all, g_all);
}

// Vacuum dynamics nodes: GV_PARTS threads per node, a warp per part (jobs.h: dyn_noair_part).  A block is GV_PARTS
// warps = 32 nodes; phase A stages each node's shared values in shared memory, one barrier, phase B.
#define GV_THREADS (32 * GV_PARTS)
#ifndef GV_MIN_BLOCKS
#define GV_MIN_BLOCKS 5 /* 96 registers, no spills; 4 (113 registers) measured slower, 6 spills (profiles/r05b_ab.txt) */
#endif
__global__ void __launch_bounds__(GV_THREADS, GV_MIN_BLOCKS)
k_jacobian_noair(const __grid_constant__ PlanView P, const int first, const int count, const int n_scen,
                 const int32_t* __restrict__ scen_ids, const double* __restrict__ x_all, double* __restrict__ out_all,
                 double* __restrict__ g_all) {
  const int per = (count + 31) / 32;  // blocks per scenario
  const int scen = blockIdx.x / per;
  const int lane = threadIdx.x & 31, part = threadIdx.x >> 5;
  const int k = (blockIdx.x - scen * per) * 32 + lane;
  __shared__ NoairStage stage[32];  // per node: what its four parts share
  const double* x = x_all + (size_t)scen * P.n_vars;
  double* out = out_all + (size_t)scen * (size_t)(P.packed ? P.n_pack : P.n_vals);
  double* g = g_all ? g_all + (size_t)scen * P.n_rows : nullptr;
  const int sid = scen_ids ? scen_ids[scen] : scen;
  const bool live = k < count;
  NodeRef nr;
  if (live) {
    nr = jac_node(P, first + k);
    dyn_noair_stage(P, sid, x, nr, part, stage[lane]);
  }
  __syncthreads();
  if (live) dyn_noair_part(P, sid, x, out, g, nr, part, stage[lane]);
}

#ifndef GR_MIN_BLOCKS
#define GR_MIN_BLOCKS 8 /* 64 registers; measured best of 5, 8, 10 (profiles/r01g_ab.txt) */
#endif
__global__ void __launch_bounds__(GR_THREADS, GR_MIN_BLOCKS)
k_residuals(const __grid_constant__ PlanView P, const int32_t* __restrict__ block_table, const int n_scen,
            const int32_t* __restrict__ scen_ids, const double* __restrict__ x_all, double* __restrict__ g_all) {
  __shared__ ResScratch sm;
  const int scen = blockIdx.x % n_scen;
  const int32_t* bt = block_table + (size_t)(blockIdx.x / n_scen) * BT_COLS;
  const double* x = x_all + (size_t)scen * P.n_vars;
  double* g = g_all + (size_t)scen * P.n_rows;
  const int sid = scen_ids ? scen_ids[scen] : scen;
  const bool dyn = bt[BT_ROLE] == BR_DYN;
  if (dyn) {
    res_block_phase0(P, sid, bt, x, threadIdx.x, sm);
    __syncthreads();
  }
  res_block_phase1(P, sid, bt, x, g, threadIdx.x, sm);
  if (dyn) {
    __syncthreads();
    res_block_phase2(P, sid, bt, x, g, threadIdx.x, GR_THREADS, sm);
  }
}

// packed[scen][i] = vals[scen][idx[i]]: the x-dependent slots, gathered for the PCIe copy of update mode
__global__ void k_pack_xdep(const double* __restrict__ vals_all, const int64_t* __restrict__ idx, long long n_xdep,
                            long long n_vals, double* __restrict__ packed_all) {
  const int scen = blockIdx.y;
  const double* vals = vals_all + (size_t)scen * n_vals;
  double* packed = packed_all + (size_t)scen * n_xdep;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_xdep; i += (long long)gridDim.x * blockDim.x)
    packed[i] = vals[idx[i]];
}

// update mode, zero-copy flavour: the x-dependent slots written straight into the caller's page-locked
// (device-mapped) host buffer over PCIe; runs of consecutive slots coalesce into full-width writes
__global__ void k_scatter_xdep_host(const double* __restrict__ vals_all, const int64_t* __restrict__ idx,
                                    long long n_xdep, long long n_vals, double* __restrict__ host_vals_all) {
  const int scen = blockIdx.y;
  const double* vals = vals_all + (size_t)scen * n_vals;
  double* host = host_vals_all + (size_t)scen * n_vals;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_xdep; i += (long long)gridDim.x * blockDim.x) {
    const long long k = idx[i];
    host[k] = vals[k];
  }
}

// Central differences (DESIGN.md H6): `out` holds the +h pass in its own layout, `minus` the -h pass packed
// ([n_scen][n_pack]).  Packed output (full == NULL): out[scen][i] = fd_central(out[scen][i], minus[scen][i]), i < n_ent
// = n_pack.  COO output: the packed map, vals[scen][full[i]] = fd_central(vals[scen][full[i]], sgn[i] * minus[scen][src[i]]),
// i < n_ent = n_xdep.
__global__ void k_fd_central(double* __restrict__ out_all, long long out_stride, const double* __restrict__ minus_all,
                             long long n_pack, int n_scen, const int64_t* __restrict__ full, const int64_t* __restrict__ src,
                             const double* __restrict__ sgn, long long n_ent) {
  for (int scen = blockIdx.y; scen < n_scen; scen += gridDim.y) {
    double* out = out_all + (size_t)scen * out_stride;
    const double* minus = minus_all + (size_t)scen * n_pack;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_ent; i += (long long)gridDim.x * blockDim.x) {
      if (full) {
        const long long k = full[i];
        out[k] = fd_central(out[k], sgn[i] * minus[src[i]]);
      } else {
        out[i] = fd_central(out[i], minus[i]);
      }
    }
  }
}

// Mesh error estimate (mesh_error.h; DESIGN.md section 11), two launches.  First one thread per (scenario, test point):
// the interpolated state and the right-hand side there, MESH_PT doubles per point into pts[n_scen][n_pts][MESH_PT].
// Then one thread per (scenario, section, state component) over the section's intervals (ints[int0[sec] ..
// int0[sec + 1])): per interval the integral and the two maxima into err_int[n_scen][n_int][11], their max into
// err[n_scen][S][11]; either output may be NULL.  INTERVALS == false (a grid without interval tables): interval sec is
// the whole section, and the kernel reads no interval list -- the loads before the first integral are those of the
// estimate without intervals.
#define GM_THREADS 128
__global__ void __launch_bounds__(GM_THREADS)
k_mesh_points(const __grid_constant__ PlanView P, const MeshPt* __restrict__ pt, const MeshSec* __restrict__ ms,
              const double* __restrict__ pool, int n_pts, int n_scen, const double* __restrict__ x_all,
              double* __restrict__ pts_all) {
  const long long i = (long long)blockIdx.x * GM_THREADS + threadIdx.x;
  if (i >= (long long)n_pts * n_scen) return;
  const int scen = (int)(i / n_pts), k = (int)(i - (long long)scen * n_pts);
  const MeshPt q = pt[k];
  const MeshTabs tb = mesh_tabs(pool, ms[q.sec], P.sec_i32[q.sec * GS_I32_COLS + GS_N]);
  double* out = pts_all + (size_t)i * MESH_PT;
  mesh_point(P, scen, x_all + (size_t)scen * P.n_vars, q.sec, tb, q.l, out, out + MESH_STATE);
}
template <bool INTERVALS>
__global__ void __launch_bounds__(GM_THREADS)
k_mesh_error(const __grid_constant__ PlanView P, const MeshSec* __restrict__ ms, const MeshInt* __restrict__ ints,
             const int32_t* __restrict__ int0, const double* __restrict__ pool, int n_pts, int n_int, int n_scen,
             const double* __restrict__ x_all, const double* __restrict__ pts_all, double* __restrict__ err_all,
             double* __restrict__ err_int) {
  const long long i = (long long)blockIdx.x * GM_THREADS + threadIdx.x;
  const int per = P.S * MESH_STATE;
  if (i >= (long long)per * n_scen) return;
  const int scen = (int)(i / per), r = (int)(i - (long long)scen * per);
  const int sec = r / MESH_STATE, c = r - sec * MESH_STATE;
  const MeshSec s = ms[sec];
  const MeshTabs tb = mesh_tabs(pool, s, P.sec_i32[sec * GS_I32_COLS + GS_N]);
  const double* pts = pts_all + ((size_t)scen * n_pts + s.pt0) * MESH_PT;
  const double* x = x_all + (size_t)scen * P.n_vars;
  const int k0 = INTERVALS ? int0[sec] : sec, k1 = INTERVALS ? int0[sec + 1] : sec + 1;
  double e = 0.0;
  for (int k = k0; k < k1; k++) {
    const double ek = mesh_component(P, x, sec, tb, s.m, pts, c, INTERVALS ? ints[k] : MeshInt{0, 0, s.m});
    if (err_int) err_int[((size_t)scen * n_int + k) * MESH_STATE + c] = ek;
    e = k == k0 ? ek : mesh_max(e, ek);
  }
  if (err_all) err_all[i] = e;
}

// Path check (mesh_error.h; DESIGN.md section 11), two launches on the same grid.  First one thread per (scenario, test
// point of an aero job over a whole section): the residual 1 - f there into r[n_scen][n_pts].  Then one thread per
// (scenario, aero job): its minimum and the test point of the minimum, res / at [n_scen][n_aero].
__global__ void __launch_bounds__(GM_THREADS)
k_path_points(const __grid_constant__ PlanView P, const PathPt* __restrict__ pt, const MeshSec* __restrict__ ms,
              const double* __restrict__ pool, int n_pts, int n_scen, const double* __restrict__ x_all,
              double* __restrict__ r_all) {
  const long long i = (long long)blockIdx.x * GM_THREADS + threadIdx.x;
  if (i >= (long long)n_pts * n_scen) return;
  const int scen = (int)(i / n_pts), k = (int)(i - (long long)scen * n_pts);
  const PathPt q = pt[k];
  const int sec = P.aero_i32[q.job * GA_I32_COLS + GA_SECTION];
  const MeshTabs tb = mesh_tabs(pool, ms[sec], P.sec_i32[sec * GS_I32_COLS + GS_N]);
  r_all[i] = mesh_path_point(P, scen, x_all + (size_t)scen * P.n_vars, q.job, tb, q.l);
}
__global__ void __launch_bounds__(GM_THREADS)
k_path_min(int n_aero, const int32_t* __restrict__ job0, int n_pts, int n_scen, const double* __restrict__ r_all,
           double* __restrict__ res_all, int32_t* __restrict__ at_all) {
  const long long i = (long long)blockIdx.x * GM_THREADS + threadIdx.x;
  if (i >= (long long)n_aero * n_scen) return;
  const int scen = (int)(i / n_aero), j = (int)(i - (long long)scen * n_aero);
  const int p0 = job0[j];
  mesh_path_min(r_all + (size_t)scen * n_pts + p0, job0[j + 1] - p0, res_all + i, at_all + i);
}

// Path rows (mesh_error.h; DESIGN.md section 11): `lanes` threads per (scenario, row).  lanes == PATH_LANES: lane 0
// evaluates the centre f and writes g = 1 - f (g_all != NULL); it reaches lanes 1-12 by a half-warp shuffle, and each
// of those writes its quotient's entries into vals[n_scen][n_vals].  lanes == 1 (residual only): the centres alone.
#define GP_THREADS 128
__global__ void __launch_bounds__(GP_THREADS)
k_path_rows(const __grid_constant__ PlanView P, const PathRow* __restrict__ rows, const MeshSec* __restrict__ ms,
            const double* __restrict__ pool, int n_rows, long long n_vals, int n_scen, int lanes, int central, double step,
            const double* __restrict__ x_all, double* __restrict__ g_all, double* __restrict__ vals_all) {
  const long long i = (long long)blockIdx.x * GP_THREADS + threadIdx.x;
  const long long item = i / lanes;
  const int lane = (int)(i - item * lanes);
  const bool live = item < (long long)n_rows * n_scen;
  const int scen = live ? (int)(item / n_rows) : 0;
  const int k = live ? (int)(item - (long long)scen * n_rows) : 0;
  const PathRow pr = rows[k];
  const int sec = P.aero_i32[pr.job * GA_I32_COLS + GA_SECTION], n = P.sec_i32[sec * GS_I32_COLS + GS_N];
  const MeshTabs tb = mesh_tabs(pool, ms[sec], n);
  const double* x = x_all + (size_t)scen * P.n_vars;
  double v[10];
  mesh_path_state(P, x, sec, tb, pr.l, v);
  double f0 = 0.0;
  if (live && lane == 0) f0 = path_lane_f(P, scen, x, pr.job, tb, pr.l, v, 0, 0.0);
  if (lanes > 1) f0 = __shfl_sync(0xffffffffu, f0, 0, PATH_LANES);  // every thread of the warp is here
  if (!live) return;
  if (lane == 0) {
    if (g_all) g_all[item] = 1.0 - f0;
    return;
  }
  if (lane > 12 || (pr.off[PR_QUAT] < 0 && lane >= 7 && lane <= 10)) return;
  const double q = path_lane_quot(P, scen, x, pr.job, tb, pr.l, v, lane, f0, central, step);
  path_lane_store(pr, tb.P + (long long)pr.l * (n + 1), n, lane, q, vals_all + (size_t)scen * n_vals);
}

// Result-table user constraints (user_table.h): one warp per (scenario, table job), lane l evaluating output_row on
// its state once; per constraint row the quotients against lane 0 come from a shuffle.  out_all == NULL: residual only
// (the pristine lane alone); g_all == NULL: Jacobian only.  Every thread of a warp reaches the shuffles (a warp is one
// job; the warps past the last job run job 0 with every lane idle).
#define GT_THREADS 128
__global__ void __launch_bounds__(GT_THREADS)
k_user_table(const __grid_constant__ PlanView P, const __grid_constant__ TabView T, const int n_scen,
             const int32_t* __restrict__ scen_ids, const double* __restrict__ x_all, double* __restrict__ out_all,
             double* __restrict__ g_all) {
  const long long w = ((long long)blockIdx.x * GT_THREADS + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const bool live = w < (long long)T.n_tab * n_scen;
  const int scen = live ? (int)(w / T.n_tab) : 0;
  const int job = live ? (int)(w - (long long)scen * T.n_tab) : 0;
  const bool active = live && (lane < GT_PRISTINE ? out_all != nullptr : (lane == GT_PRISTINE && g_all != nullptr));
  const int sid = scen_ids ? scen_ids[scen] : scen;
  double out[GO_COLS];
  if (active) table_lane_eval(P, T, sid, x_all + (size_t)scen * P.n_vars, job, lane, out);
  double* vals = out_all ? out_all + (size_t)scen * (size_t)(P.packed ? P.n_pack : P.n_vals) : nullptr;
  double* g = g_all ? g_all + (size_t)scen * P.n_rows : nullptr;
  const int nrow = T.i32[(long long)job * GT_I32_COLS + GT_NROW];
  for (int r = 0; r < nrow; r++) {
    const double v = active ? table_row_value(T, job, r, out) : 0.0;
    const double v0 = __shfl_sync(0xffffffffu, v, 0);
    if (active) table_lane_store(P, T, job, r, lane, v, v0, vals, g);
  }
}

// probe: is a*b+c left unfused?  (1 + 2^-30)(1 - 2^-30) - 1 is 0 unfused, -2^-60 fused
__global__ void k_unfused_probe(double a, double b, double c, double* out) { *out = a * b + c; }

// FP64 issue-rate probes (DESIGN.md H9)
__global__ void k_fp64_fma(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
         a7 = a0 + 7;
  const double b = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; i++) {
    a0 = __fma_rn(a0, b, c); a1 = __fma_rn(a1, b, c); a2 = __fma_rn(a2, b, c); a3 = __fma_rn(a3, b, c);
    a4 = __fma_rn(a4, b, c); a5 = __fma_rn(a5, b, c); a6 = __fma_rn(a6, b, c); a7 = __fma_rn(a7, b, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}
__global__ void k_fp64_muladd(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
         a7 = a0 + 7;
  const double b = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; i++) {
    a0 = __dadd_rn(__dmul_rn(a0, b), c); a1 = __dadd_rn(__dmul_rn(a1, b), c);
    a2 = __dadd_rn(__dmul_rn(a2, b), c); a3 = __dadd_rn(__dmul_rn(a3, b), c);
    a4 = __dadd_rn(__dmul_rn(a4, b), c); a5 = __dadd_rn(__dmul_rn(a5, b), c);
    a6 = __dadd_rn(__dmul_rn(a6, b), c); a7 = __dadd_rn(__dmul_rn(a7, b), c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CU(call)                                                                                  \
  do {                                                                                            \
    cudaError_t e_ = (call);                                                                      \
    if (e_ != cudaSuccess)                                                                        \
      return fail(GELATO_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));           \
  } while (0)

using gelato_host::DeviceBuf;
using gelato_host::Event;
using gelato_host::GraphExec;
using gelato_host::PinnedBuf;
using gelato_host::Stream;

// a test grid on the device (gelato_plan_set_mesh_grid, gelato_plan_set_path_rows): its sections and table pool
struct TestGrid {
  DeviceBuf<MeshSec> sec;
  DeviceBuf<double> pool;
};

struct GelatoPlan {
  int device = 0;
  PlanView view{};         // device pointers
  PlanView shared_view{};  // the view as created, with the blocks every scenario shares (gelato_plan_set_scenarios)
  std::vector<DeviceBuf<char>> owned;
  int32_t* jac_blocks = nullptr;  // n_jac_main dynamics / aero / event blocks (roles interleaved), then the linear-row blocks
  int n_jac_blocks = 0, n_jac_main = 0;
  int32_t *jac_heavy = nullptr, *jac_light = nullptr;  // the same blocks by role group (measurements)
  int n_jac_heavy = 0, n_jac_light = 0;
  int vac_first = 0, n_vac = 0;  // vacuum dynamics nodes: k_jacobian_noair, one thread per node
  int32_t* res_blocks = nullptr;
  int n_res_blocks = 0;
  // packed output (plan_host.h: build_packed_layout)
  long long n_pack = 0;
  std::vector<int64_t> pk_full, pk_src;
  std::vector<double> pk_sgn;
  std::vector<DeviceBuf<char>> scen_owned;  // uploads of gelato_plan_set_scenarios (replaced by the next call)
  const double* vals_template = nullptr;    // [n_vals] (or [n_scen][n_vals])
  const double* shared_template = nullptr;  // the plan's own [n_vals]
  long long vals_template_sstride = 0;
  int n_scen_cfg = 1;
  // staging of every host-buffer entry point: x, g and the scenario ids of the batch slots, which hold either the
  // caller's ids or 0, 1, 2 ... (ids_iota); the outputs of a diagnostic on a test grid (eval_diag), at most two a call
  DeviceBuf<double> d_x, d_g;
  PinnedBuf<double> h_x, h_g;
  DeviceBuf<char> d_diag[2];
  PinnedBuf<char> h_diag[2];
  DeviceBuf<int32_t> d_ids;
  bool ids_iota = false;
  // COO Jacobian of the host entry points: slot k of d_vals holds scenario k's constants for k < vals_filled (written
  // once, the kernels only rewrite x-dependent slots); d_vals_ids holds those of the slots of an _ids call
  DeviceBuf<double> d_vals, d_vals_ids;
  size_t vals_filled = 0;
  PinnedBuf<double> h_vals;
  // packed host entry points
  DeviceBuf<double> d_packed;
  PinnedBuf<double> h_packed;
  // small host-buffer objfunc calls: upload, kernel and download as ONE captured graph launch (the staging pointers
  // and the plan view are baked into it: rebuilt whenever either changes)
  GraphExec res_graph;
  int res_graph_n = 0;
  // update mode
  const int64_t* d_xdep = nullptr;
  std::vector<int64_t> h_xdep;
  long long n_xdep = 0;
  DeviceBuf<double> d_pack;  // [n_scen][n_xdep]
  PinnedBuf<double> h_pack;
  int host_threads = 0;
  // scattered slots of a page-locked caller buffer: packed + host pool (0) or written from the device (1).
  // With 8+ host threads the pool is 1.6x faster end to end (profiles/r01v_e2e.txt); few cores: zero-copy.
  int update_zero_copy = std::thread::hardware_concurrency() < 8 ? 1 : 0;
  std::vector<std::pair<int64_t, int64_t>> big_runs;  // (first slot, length) of the long runs in xdep_idx
  const int64_t* d_xdep_small = nullptr;              // the slots outside those runs
  std::vector<int64_t> h_small;
  long long n_small = 0;
  // The plan's streams.  Lane 0 is created with the plan and serves every call (a device-pointer call launches on the
  // caller's stream with lane 0's side stream and events); the host-buffer entry points pipeline a batch over slices,
  // slice k's upload and kernels overlapping slice k-1's copies on lane k (created on first use).
  struct Lane {
    Stream stream, copy_stream;
    Stream pair_stream;  // the vacuum-node kernel of a Jacobian evaluation, concurrent with the block kernel
    Event ev_kernel, ev_copy, ev_fork, ev_join, ev_h2d, ev_g, ev_gdone;
    std::vector<Event> chunk_ev;
  };
  std::vector<Lane> lanes;
  int update_slices = 0;  // 0 = choose from the batch size
  // finite-difference mode (gelato_plan_set_fd); central: the -h pass of batch slot s goes to d_fd + s * n_pack
  int fd_mode = GELATO_FD_FORWARD;
  double fd_step = 0.0;
  DeviceBuf<double> d_fd;
  const int64_t *d_pk_full = nullptr, *d_pk_src = nullptr;  // the packed map on the device (uploaded on first use)
  const double* d_pk_sgn = nullptr;
  // mesh error estimate (gelato_plan_set_mesh_grid): the grid and its test points on the device, n_mesh_pts = 0 until
  // a grid is set; d_mesh_pts is the per-point scratch
  std::vector<int32_t> sec_n;  // LGR nodes of each section
  TestGrid mesh_grid;
  DeviceBuf<MeshPt> d_mesh_pt;
  DeviceBuf<double> d_mesh_pts;
  int n_mesh_pts = 0;
  // its intervals, and each section's first one (d_mesh_int0[S + 1]); n_mesh_int intervals in all; mesh_intervals:
  // the grid came with interval tables (else interval i is section i)
  DeviceBuf<MeshInt> d_mesh_int;
  DeviceBuf<int32_t> d_mesh_int0;
  int n_mesh_int = 0;
  bool mesh_intervals = false;
  // path check on the same grid: the test points of the aero jobs over a whole section and each job's first one
  // (plan_host.h: build_path_points, rebuilt with the grid), the per-point scratch d_path_r
  std::vector<int32_t> aero_i32;  // the aero jobs, as the plan description gave them
  DeviceBuf<PathPt> d_path_pt;
  DeviceBuf<int32_t> d_path_job0;
  DeviceBuf<double> d_path_r;
  int n_path_pts = 0;
  // path rows (gelato_plan_set_path_rows) on a grid of their own: the grid, the row list (plan_host.h: build_path_rows)
  // on the host and the device, and the values per scenario
  bool prow_set = false;
  std::vector<PathRow> prow;
  long long prow_vals = 0;
  TestGrid prow_grid;
  DeviceBuf<PathRow> d_prow;
  // result-table user constraints (user_table.h; tab.n_tab = 0: none, and nothing is launched for them)
  TabView tab{};
  long long launches = 0;
  Event ev0, ev1;
};
typedef GelatoPlan::Lane Lane;

template <typename T>
static int upload(std::vector<DeviceBuf<char>>& owner, const T* src, size_t count, const T** dst) {
  *dst = nullptr;
  if (count == 0 || src == nullptr) return GELATO_OK;
  owner.emplace_back();
  CU(owner.back().reserve(count * sizeof(T)));
  CU(cudaMemcpy(owner.back().get(), src, count * sizeof(T), cudaMemcpyHostToDevice));
  *dst = reinterpret_cast<const T*>(owner.back().get());
  return GELATO_OK;
}

static int add_lane(GelatoPlan* p) {
  p->lanes.emplace_back();
  Lane& L = p->lanes.back();
  for (cudaStream_t* st : {L.stream.out(), L.copy_stream.out(), L.pair_stream.out()})
    CU(cudaStreamCreateWithFlags(st, cudaStreamNonBlocking));
  for (cudaEvent_t* e : {L.ev_kernel.out(), L.ev_copy.out(), L.ev_fork.out(), L.ev_join.out(), L.ev_h2d.out(), L.ev_g.out(),
                         L.ev_gdone.out()})
    CU(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  return GELATO_OK;
}

// One Jacobian evaluation: the block kernel (air dynamics nodes, aero rows, fallback nodes, event rows) on `st` and the
// one-thread-per-node kernel of the vacuum nodes on the lane's pair stream, forked from and joined back into `st` with
// the lane's two events.
// g_dev != NULL: pair evaluation -- both also write objfunc's rows (collocation defects of their nodes, aero / event
// rows at the pristine state) and the linear-row blocks at the end of the block table are launched too.
// packed: output layout.
// (Variants measured and dropped: phase 0 as its own launch with pp | rq | q staged through L2, 38 % slower,
// profiles/r01i_split_ab.txt; the vacuum nodes as blocks of the block kernel, 0.084 ms instead of 0.03,
// profiles/r02_probe.txt.)
// A sub-range of the evaluation (one problem sharded over GPUs): blocks [b0, b0 + nb) of the block table and vacuum
// nodes [v0, v0 + nv) of the vacuum list; nb < 0: everything.
struct JacRange {
  int b0 = 0, nb = -1, v0 = 0, nv = 0;
};
// The table jobs of n_scen batch slots on `st` (nothing for a plan without them): view v's layout and step, out_dev
// NULL for a residual evaluation, g_dev NULL for a Jacobian-only one.
static int launch_table(GelatoPlan* p, const PlanView& v, const double* x_dev, double* out_dev, double* g_dev, int n_scen,
                        const int32_t* ids_dev, cudaStream_t st) {
  if (p->tab.n_tab == 0) return GELATO_OK;
  const long long threads = (long long)p->tab.n_tab * n_scen * 32;
  k_user_table<<<(unsigned)((threads + GT_THREADS - 1) / GT_THREADS), GT_THREADS, 0, st>>>(v, p->tab, n_scen, ids_dev, x_dev,
                                                                                          out_dev, g_dev);
  p->launches++;
  CU(cudaGetLastError());
  return GELATO_OK;
}

// dx: the step of the finite-difference protocol (the plan's dx for forward differences).
// The table jobs go on the pair stream next to the block kernel; a sub-range evaluates them when it starts at block 0.
static int launch_jacobian_pass(GelatoPlan* p, double dx, const double* x_dev, double* out_dev, double* g_dev, int n_scen,
                                cudaStream_t st, const Lane& L, const int32_t* ids_dev, bool packed, JacRange rg = JacRange()) {
  PlanView v = p->view;
  v.packed = packed ? 1 : 0;
  v.un.dx = dx;
  const bool all = rg.nb < 0;
  const int nb = all ? (g_dev ? p->n_jac_blocks : p->n_jac_main) : rg.nb;
  const int nv = all ? p->n_vac : rg.nv;
  const int v_first = p->vac_first + (all ? 0 : rg.v0);
  const int32_t* table = p->jac_blocks + (size_t)(all ? 0 : rg.b0) * BT_COLS;
  const cudaStream_t aux = L.pair_stream;
  const bool tab = p->tab.n_tab > 0 && (all || (rg.b0 == 0 && rg.nb > 0));
  const bool side = (nv > 0 || tab) && nb > 0 && aux != st;
  if (side) {
    CU(cudaEventRecord(L.ev_fork, st));
    CU(cudaStreamWaitEvent(aux, L.ev_fork, 0));
  }
  if (nv > 0) {
    const int per = (nv + 31) / 32;
    k_jacobian_noair<<<(unsigned)per * n_scen, GV_THREADS, 0, side ? aux : st>>>(v, v_first, nv, n_scen, ids_dev, x_dev, out_dev,
                                                                                g_dev);
    p->launches++;
  }
  if (tab) {
    int rc = launch_table(p, v, x_dev, out_dev, g_dev, n_scen, ids_dev, side ? aux : st);
    if (rc) return rc;
  }
  if (nb > 0) {
    k_jacobian<<<(unsigned)nb * n_scen, GJ_THREADS, 0, st>>>(v, table, n_scen, ids_dev, x_dev, out_dev, g_dev);
    p->launches++;
  }
  CU(cudaGetLastError());
  if (side) {
    CU(cudaEventRecord(L.ev_join, aux));
    CU(cudaStreamWaitEvent(st, L.ev_join, 0));
  }
  return GELATO_OK;
}

// The central-difference scratch for batch slots [0, n_scen) and the packed map on the device; nothing in forward mode.
// Every entry point that evaluates the Jacobian calls it before its first launch.
static int ensure_fd_scratch(GelatoPlan* p, size_t n_scen) {
  if (p->fd_mode != GELATO_FD_CENTRAL) return GELATO_OK;
  CU(cudaSetDevice(p->device));
  if (!p->d_pk_full && !p->pk_full.empty()) {
    int rc;
    if ((rc = upload(p->owned, p->pk_full.data(), p->pk_full.size(), &p->d_pk_full)) != GELATO_OK) return rc;
    if ((rc = upload(p->owned, p->pk_src.data(), p->pk_src.size(), &p->d_pk_src)) != GELATO_OK) return rc;
    if ((rc = upload(p->owned, p->pk_sgn.data(), p->pk_sgn.size(), &p->d_pk_sgn)) != GELATO_OK) return rc;
  }
  CU(p->d_fd.reserve(std::max<size_t>(1, n_scen * (size_t)p->n_pack)));  // synchronises: no launch still reads the old region
  return GELATO_OK;
}

// One Jacobian evaluation in the plan's finite-difference mode (DESIGN.md H6).  Forward: one pass with the plan's dx.
// Central: the +h pass writes the caller's output (and g of a pair evaluation), the -h pass (Jacobian only) writes the
// packed scratch of batch slots [s0, s0 + n_scen) -- slices of one batch in flight on several streams use disjoint
// regions -- and k_fd_central averages the two into the caller's output.
static int launch_jacobian(GelatoPlan* p, const double* x_dev, double* out_dev, double* g_dev, int n_scen, cudaStream_t st,
                           const Lane& L, const int32_t* ids_dev, bool packed, int s0 = 0) {
  if (p->fd_mode != GELATO_FD_CENTRAL)
    return launch_jacobian_pass(p, p->view.un.dx, x_dev, out_dev, g_dev, n_scen, st, L, ids_dev, packed);
  if (((size_t)s0 + (size_t)n_scen) * p->n_pack > p->d_fd.size())
    return fail(GELATO_ERR_ARG, "central-difference scratch not allocated");
  const double h = p->fd_step;
  double* minus = p->d_fd.get() + (size_t)s0 * p->n_pack;
  int rc = launch_jacobian_pass(p, h, x_dev, out_dev, g_dev, n_scen, st, L, ids_dev, packed);
  if (rc) return rc;
  if ((rc = launch_jacobian_pass(p, -h, x_dev, minus, nullptr, n_scen, st, L, ids_dev, true))) return rc;
  const long long n_ent = packed ? p->n_pack : (long long)p->pk_full.size();
  if (n_ent == 0) return GELATO_OK;
  const int threads = 256;
  const unsigned bx = (unsigned)std::min<long long>((n_ent + threads - 1) / threads, 4096);
  const unsigned by = (unsigned)std::min(n_scen, 65535);
  k_fd_central<<<dim3(bx, by), threads, 0, st>>>(out_dev, packed ? p->n_pack : p->view.n_vals, minus, p->n_pack, n_scen,
                                                 packed ? nullptr : p->d_pk_full, p->d_pk_src, p->d_pk_sgn, n_ent);
  p->launches++;
  CU(cudaGetLastError());
  return GELATO_OK;
}

static int launch_residuals(GelatoPlan* p, const double* x_dev, double* g_dev, int n_scen, const int32_t* ids_dev,
                            cudaStream_t st) {
  k_residuals<<<(unsigned)p->n_res_blocks * n_scen, GR_THREADS, 0, st>>>(p->view, p->res_blocks, n_scen, ids_dev, x_dev, g_dev);
  p->launches++;
  CU(cudaGetLastError());
  return launch_table(p, p->view, x_dev, nullptr, g_dev, n_scen, ids_dev, st);
}

static void drop_graph(GelatoPlan* p) {
  p->res_graph.reset();
  p->res_graph_n = 0;
}

extern "C" {

const char* gelato_last_error(void) { return g_err.c_str(); }
void gelato_set_error_(const char* msg) { g_err = msg ? msg : ""; }  // for leaf_api.cu

int gelato_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int gelato_plan_create(const GelatoPlanDesc* d, int device, GelatoPlan** out) {
  if (!d || !out) return fail(GELATO_ERR_ARG, "null argument");
  if (const char* why = validate_desc(d)) return fail(GELATO_ERR_ARG, why);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(GELATO_ERR_CUDA, "no CUDA device: the B200 kernels are the only evaluation path (no CPU fallback)");
  CU(cudaSetDevice(device));
  std::unique_ptr<GelatoPlan> p(new GelatoPlan());
  p->device = device;
  PlanView& v = p->view;
  planview_scalars(d, v);
  const int S = v.S;
  int rc;
#define UP(dst, src, count) if ((rc = upload(p->owned, src, (size_t)(count), &(dst))) != GELATO_OK) return rc;
  for (int i = 0; i < S; i++) p->sec_n.push_back(d->sec_i32[i * GS_I32_COLS + GS_N]);
  if (d->n_aero > 0) p->aero_i32.assign(d->aero_i32, d->aero_i32 + (size_t)d->n_aero * GA_I32_COLS);
  UP(v.sec_i32, d->sec_i32, (size_t)S * GS_I32_COLS)
  UP(v.sec_i64, d->sec_i64, (size_t)S * GS_I64_COLS)
  UP(v.sec_f64, d->sec_f64, (size_t)S * GS_F64_COLS)
  UP(v.d_pool, d->d_pool, d->d_pool_len)
  UP(v.tau_pool, d->tau_pool, d->tau_pool_len)
  UP(v.wind, d->wind, (size_t)d->n_wind * 3)
  UP(v.ca, d->ca, (size_t)d->n_ca * 2)
  UP(v.lin_i32, d->lin_i32, (size_t)d->n_lin * GL_I32_COLS)
  UP(v.lin_f64, d->lin_f64, (size_t)d->n_lin * GL_F64_COLS)
  UP(v.aero_i32, d->aero_i32, (size_t)d->n_aero * GA_I32_COLS)
  UP(v.aero_i64, d->aero_i64, (size_t)d->n_aero * GA_I64_COLS)
  UP(v.aero_f64, d->aero_f64, (size_t)d->n_aero * GA_F64_COLS)
  UP(v.rc_aero, d->rc_aero, d->rc_aero ? (size_t)v.n_vars : 0)
  UP(v.evt_i32, d->evt_i32, (size_t)d->n_evt * GE_I32_COLS)
  UP(v.evt_i64, d->evt_i64, (size_t)d->n_evt * GE_I64_COLS)
  UP(v.evt_f64, d->evt_f64, (size_t)d->n_evt * GE_F64_COLS)
  if (d->xdep_idx && d->n_xdep > 0) {
    for (int64_t i = 0; i < d->n_xdep; i++)
      if (d->xdep_idx[i] < 0 || d->xdep_idx[i] >= d->n_vals || (i > 0 && d->xdep_idx[i] <= d->xdep_idx[i - 1]))
        return fail(GELATO_ERR_ARG, "xdep_idx must be strictly ascending and inside [0, n_vals)");
    p->h_xdep.assign(d->xdep_idx, d->xdep_idx + d->n_xdep);
    p->n_xdep = d->n_xdep;
    UP(p->d_xdep, d->xdep_idx, d->n_xdep)
    // split for the zero-copy route: long runs of consecutive slots go through the copy engine (one strided
    // 2-D copy per run covers every scenario), the scattered rest is written by a kernel
    std::vector<int64_t> small;
    for (int64_t i = 0; i < d->n_xdep;) {
      int64_t j = i + 1;
      while (j < d->n_xdep && d->xdep_idx[j] == d->xdep_idx[j - 1] + 1) j++;
      if (j - i >= 512) p->big_runs.push_back({d->xdep_idx[i], j - i});
      else small.insert(small.end(), d->xdep_idx + i, d->xdep_idx + j);
      i = j;
    }
    p->n_small = (long long)small.size();
    p->h_small = small;
    UP(p->d_xdep_small, small.data(), small.size())
  }
  UP(p->vals_template, d->vals_template, d->n_vals)
  p->shared_template = p->vals_template;
  p->tab.n_tab = d->n_tab;
  if (d->n_tab > 0) {
    UP(p->tab.i32, d->tab_i32, (size_t)d->n_tab * GT_I32_COLS)
    UP(p->tab.f64, d->tab_f64, (size_t)d->n_tab * GT_F64_COLS)
    UP(p->tab.col, d->tab_col, d->n_tab_rows)
    UP(p->tab.aux, d->tab_aux, d->n_tab_rows)
    UP(p->tab.sf, d->tab_sf, (size_t)d->n_tab_rows * GT_SF_COLS)
  }

  // block tables
  HostTables ht;
  build_host_tables(d, ht);
  p->n_jac_blocks = (int)(ht.jac_blocks.size() / BT_COLS);
  p->n_res_blocks = (int)(ht.res_blocks.size() / BT_COLS);
  p->n_jac_main = ht.n_jac_main;
  p->vac_first = ht.vac_first;
  p->n_vac = ht.n_vac;
  p->n_jac_heavy = (int)(ht.jac_heavy.size() / BT_COLS);
  p->n_jac_light = (int)(ht.jac_light.size() / BT_COLS);
  const int32_t* tb = nullptr;
  UP(tb, ht.jac_heavy.data(), ht.jac_heavy.size())
  p->jac_heavy = const_cast<int32_t*>(tb);
  UP(tb, ht.jac_light.data(), ht.jac_light.size())
  p->jac_light = const_cast<int32_t*>(tb);
  {
    PackedLayout L;
    build_packed_layout(d, L);
    if (d->xdep_idx && d->n_xdep > 0 &&
        ((size_t)d->n_xdep != L.full_slot.size() || !std::equal(L.full_slot.begin(), L.full_slot.end(), d->xdep_idx)))
      return fail(GELATO_ERR_ARG, "xdep_idx is not the set of slots the Jacobian kernel writes for this plan");
    p->n_pack = L.n_pack;
    v.n_pack = L.n_pack;
    UP(v.sec_pk, L.sec_pk.data(), L.sec_pk.size())
    UP(v.aero_pk, L.aero_pk.data(), L.aero_pk.size())
    UP(v.evt_pk, L.evt_pk.data(), L.evt_pk.size())
    UP(p->tab.pk, L.tab_pk.data(), L.tab_pk.size())
    p->pk_full.swap(L.full_slot);
    p->pk_src.swap(L.src);
    p->pk_sgn.swap(L.sgn);
  }
  UP(tb, ht.jac_blocks.data(), ht.jac_blocks.size())
  p->jac_blocks = const_cast<int32_t*>(tb);
  UP(tb, ht.res_blocks.data(), ht.res_blocks.size())
  p->res_blocks = const_cast<int32_t*>(tb);
  UP(v.node_rec, ht.node_rec.data(), ht.node_rec.size())
  UP(v.jac_rec, ht.jac_rec.data(), ht.jac_rec.size())
  UP(v.aero_rows, ht.aero_rows.data(), ht.aero_rows.size())
#undef UP
  v.n_aero_rows = (int)ht.aero_rows.size();
  p->shared_view = v;

  if ((rc = add_lane(p.get()))) return rc;
  CU(cudaEventCreate(p->ev0.out()));
  CU(cudaEventCreate(p->ev1.out()));
  *out = p.release();
  return GELATO_OK;
}

int gelato_plan_set_scenarios(GelatoPlan* p, const GelatoScenarioDesc* sc) {
  if (!p || !sc || sc->n_scen <= 0) return fail(GELATO_ERR_ARG, "bad scenario descriptor");
  CU(cudaSetDevice(p->device));
  CU(cudaDeviceSynchronize());  // nothing in flight may still read the blocks being replaced
  // Every call starts from the plan's own blocks, so a NULL member means the block every scenario shares.  The blocks
  // of an earlier call are superseded as a whole.
  PlanView& v = p->view;
  v = p->shared_view;
  p->vals_template = p->shared_template;
  p->vals_template_sstride = 0;
  p->scen_owned.clear();
  p->n_scen_cfg = sc->n_scen;
  // the staging Jacobian buffer holds the constants of the PREVIOUS scenarios: have it refilled on the next call
  p->vals_filled = 0;
  drop_graph(p);
  const size_t n = (size_t)sc->n_scen;
  int rc;
  if (sc->sec_f64) {
    if ((rc = upload(p->scen_owned, sc->sec_f64, n * v.S * GS_F64_COLS, &v.sec_f64))) return rc;
    v.sec_f64_sstride = (long long)v.S * GS_F64_COLS;
  }
  if (sc->wind) {
    if ((rc = upload(p->scen_owned, sc->wind, n * v.n_wind * 3, &v.wind))) return rc;
    v.wind_sstride = (long long)v.n_wind * 3;
  }
  if (sc->unit_mass && (rc = upload(p->scen_owned, sc->unit_mass, n, &v.unit_mass_scen))) return rc;
  if (sc->lin_const && (rc = upload(p->scen_owned, sc->lin_const, n * v.n_lin, &v.lin_const_scen))) return rc;
  if (sc->vals_template) {
    if ((rc = upload(p->scen_owned, sc->vals_template, n * v.n_vals, &p->vals_template))) return rc;
    p->vals_template_sstride = v.n_vals;
  }
  return GELATO_OK;
}

int gelato_plan_destroy(GelatoPlan* p) {
  if (!p) return GELATO_OK;
  cudaSetDevice(p->device);
  delete p;
  return GELATO_OK;
}

int gelato_plan_set_fd(GelatoPlan* p, int32_t mode, double step) {
  if (!p) return fail(GELATO_ERR_ARG, "null plan");
  if (mode == GELATO_FD_FORWARD) {
    p->fd_mode = mode;
    return GELATO_OK;
  }
  if (mode != GELATO_FD_CENTRAL) return fail(GELATO_ERR_ARG, "unknown finite-difference mode");
  if (!(step > 0.0 && step <= 1e-3)) return fail(GELATO_ERR_ARG, "the central-difference step must be finite and in (0, 1e-3]");
  p->fd_mode = mode;
  p->fd_step = step;
  return GELATO_OK;
}

int gelato_plan_get_fd(const GelatoPlan* p, int32_t* mode, double* step) {
  if (!p || !mode || !step) return fail(GELATO_ERR_ARG, "null argument");
  *mode = p->fd_mode;
  *step = p->fd_mode == GELATO_FD_CENTRAL ? p->fd_step : p->view.un.dx;
  return GELATO_OK;
}

int32_t gelato_plan_n_vars(const GelatoPlan* p) { return p ? p->view.n_vars : 0; }
int32_t gelato_plan_n_rows(const GelatoPlan* p) { return p ? p->view.n_rows : 0; }
int64_t gelato_plan_n_vals(const GelatoPlan* p) { return p ? p->view.n_vals : 0; }
int64_t gelato_plan_launch_count(const GelatoPlan* p) { return p ? p->launches : 0; }
int64_t gelato_plan_n_xdep(const GelatoPlan* p) { return p ? p->n_xdep : 0; }
int32_t gelato_plan_n_blocks(const GelatoPlan* p, int which) {
  if (!p) return 0;
  switch (which) {
    case 0: return p->n_res_blocks;
    case 1: return p->n_jac_main;
    case 2: return p->n_jac_heavy;
    case 3: return p->n_jac_light;
    case 5: return p->n_vac;
    default: return p->n_jac_blocks;
  }
}

static int check_scen(GelatoPlan* p, int n_scen) {
  if (!p) return fail(GELATO_ERR_ARG, "null plan");
  if (n_scen <= 0) return fail(GELATO_ERR_ARG, "n_scen must be positive");
  const bool per_scen = p->view.sec_f64_sstride || p->view.wind_sstride || p->view.unit_mass_scen ||
                        p->view.lin_const_scen || p->vals_template_sstride;
  if (per_scen && n_scen > p->n_scen_cfg)
    return fail(GELATO_ERR_ARG, "n_scen exceeds the configured scenario blocks");
  const long long most = std::max(p->n_jac_blocks, p->n_res_blocks);
  if (most * n_scen > 0x7fffffffLL) return fail(GELATO_ERR_ARG, "blocks x n_scen exceeds the grid limit");
  return GELATO_OK;
}

// The start of every device-pointer entry point: the batch checked, the plan's device made current, and the stream to
// launch on (the caller's, else the plan's own).
static int begin_dev(GelatoPlan* p, int n_scen, void* stream, cudaStream_t* st) {
  int rc = check_scen(p, n_scen);
  if (rc) return rc;
  CU(cudaSetDevice(p->device));
  *st = stream ? (cudaStream_t)stream : p->lanes[0].stream;
  return GELATO_OK;
}

int gelato_eval_residuals_dev(GelatoPlan* p, const double* x_dev, double* g_dev, int32_t n_scen, void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  return launch_residuals(p, x_dev, g_dev, n_scen, nullptr, st);
}

int gelato_eval_pair_dev(GelatoPlan* p, const double* x_dev, double* g_dev, double* vals_dev, int32_t n_scen, void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  // objfunc's rows come out of the Jacobian launch: the dynamics blocks hold the right-hand side of the pristine
  // x as their centre column and subtract it from the D.X products; aero and event blocks carry one more column
  // at the pristine state; the linear rows are blocks of their own (no second pass over the physics)
  if ((rc = ensure_fd_scratch(p, n_scen))) return rc;
  return launch_jacobian(p, x_dev, vals_dev, g_dev, n_scen, st, p->lanes[0], nullptr, false);
}

int gelato_eval_pair_packed_dev(GelatoPlan* p, const double* x_dev, double* g_dev, double* packed_dev, int32_t n_scen,
                                void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  if ((rc = ensure_fd_scratch(p, n_scen))) return rc;
  return launch_jacobian(p, x_dev, packed_dev, g_dev, n_scen, st, p->lanes[0], nullptr, true);
}

// ONE problem sharded over GPUs (SURVEY.md 8(e)-2): the pair evaluation restricted to blocks
// [block_first, block_first + block_count) of the block table and vacuum nodes [vac_first, vac_first + vac_count).
// Every output slot and residual row belongs to exactly one block or vacuum node, so ranks with disjoint ranges that
// cover everything fill disjoint parts of the packed vector and of g.
int gelato_eval_pair_packed_range_dev(GelatoPlan* p, const double* x_dev, double* g_dev, double* packed_dev, int32_t n_scen,
                                      int32_t block_first, int32_t block_count, int32_t vac_first, int32_t vac_count,
                                      void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  if (!g_dev || !packed_dev) return fail(GELATO_ERR_ARG, "null buffer");
  if (p->fd_mode != GELATO_FD_FORWARD) return fail(GELATO_ERR_ARG, "the range evaluation supports forward differences only");
  if (block_first < 0 || block_count < 0 || block_first + block_count > p->n_jac_blocks || vac_first < 0 || vac_count < 0 ||
      vac_first + vac_count > p->n_vac)
    return fail(GELATO_ERR_ARG, "block or vacuum-node range outside the plan");
  JacRange rg;
  rg.b0 = block_first; rg.nb = block_count; rg.v0 = vac_first; rg.nv = vac_count;
  return launch_jacobian_pass(p, p->view.un.dx, x_dev, packed_dev, g_dev, n_scen, st, p->lanes[0], nullptr, true, rg);
}

int gelato_fill_template(GelatoPlan* p, double* vals_dev, int32_t n_scen, void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  if (p->vals_template_sstride) {
    CU(cudaMemcpyAsync(vals_dev, p->vals_template, (size_t)n_scen * p->view.n_vals * sizeof(double),
                       cudaMemcpyDeviceToDevice, st));
  } else {
    for (int s = 0; s < n_scen; s++)
      CU(cudaMemcpyAsync(vals_dev + (size_t)s * p->view.n_vals, p->vals_template,
                         (size_t)p->view.n_vals * sizeof(double), cudaMemcpyDeviceToDevice, st));
  }
  return GELATO_OK;
}

int gelato_eval_jacobian_dev(GelatoPlan* p, const double* x_dev, double* vals_dev, int32_t n_scen, void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  // the constants and D entries of vals_dev were put there once by gelato_fill_template;
  // the kernels rewrite every x-dependent slot and never touch the rest
  if ((rc = ensure_fd_scratch(p, n_scen))) return rc;
  return launch_jacobian(p, x_dev, vals_dev, nullptr, n_scen, st, p->lanes[0], nullptr, false);
}

// x, g and ids staging of the host-buffer entry points for n_scen batch slots.  They grow together, and the captured
// residual graph bakes in their pointers: growing them drops it.
static int ensure_staging(GelatoPlan* p, size_t n_scen) {
  const PlanView& v = p->view;
  if (n_scen <= p->d_ids.size()) return GELATO_OK;
  drop_graph(p);
  CU(p->d_x.reserve(n_scen * v.n_vars));
  CU(p->h_x.reserve(n_scen * v.n_vars));
  CU(p->d_g.reserve(n_scen * v.n_rows));
  CU(p->h_g.reserve(n_scen * v.n_rows));
  CU(p->d_ids.reserve(n_scen));
  p->ids_iota = false;
  return GELATO_OK;
}

// The COO Jacobian staging with the constants of batch slots [0, n_scen) in place.
static int ensure_vals(GelatoPlan* p, size_t n_scen) {
  if (n_scen <= p->vals_filled) return GELATO_OK;
  CU(p->d_vals.reserve(n_scen * (size_t)p->view.n_vals));
  int rc = gelato_fill_template(p, p->d_vals.get(), (int)n_scen, p->lanes[0].stream);
  if (rc) return rc;
  CU(cudaStreamSynchronize(p->lanes[0].stream));  // the other lanes' kernels write into it too
  p->vals_filled = n_scen;
  return GELATO_OK;
}

// The scenario ids of the batch slots in d_ids, uploaded on `st`: the caller's `ids` (each checked against the
// configured scenarios), else 0, 1, 2 ... when `sliced` (a slice of a batch names its scenarios), else none (*out = NULL).
static int stage_ids(GelatoPlan* p, const int32_t* ids, int n_scen, bool sliced, cudaStream_t st, const int32_t** out) {
  *out = nullptr;
  if (ids) {
    for (int k = 0; k < n_scen; k++)
      if (ids[k] < 0 || ids[k] >= p->n_scen_cfg) return fail(GELATO_ERR_ARG, "scenario id outside the configured scenarios");
    CU(cudaMemcpyAsync(p->d_ids.get(), ids, (size_t)n_scen * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    p->ids_iota = false;
  } else if (!sliced) {
    return GELATO_OK;
  } else if (!p->ids_iota) {
    std::vector<int32_t> iota(p->d_ids.size());
    for (size_t k = 0; k < iota.size(); k++) iota[k] = (int32_t)k;
    CU(cudaMemcpyAsync(p->d_ids.get(), iota.data(), iota.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    p->ids_iota = true;
  }
  *out = p->d_ids.get();
  return GELATO_OK;
}

// page-locked host memory can be DMA'd directly; pageable memory goes through the plan's staging buffers
static bool is_pinned(const void* ptr) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

// The source of the upload of a caller's x[n]: x itself when it is page-locked, else `stage` with a copy of it.
static const double* host_src(const double* x, double* stage, size_t n) {
  if (is_pinned(x)) return x;
  memcpy(stage, x, n * sizeof(double));
  return stage;
}

// The destination of the download of a caller's out[n] (out == NULL: none): out itself when it is page-locked, else
// `stage`, grown as needed; land() copies it over once the download is complete.  (Templates: C++ linkage.)
extern "C++" {
template <typename T>
static int host_dst(T* out, PinnedBuf<T>& stage, size_t n, T** dst) {
  *dst = out;
  if (!out || is_pinned(out)) return GELATO_OK;
  CU(stage.reserve(n));
  *dst = stage.get();
  return GELATO_OK;
}

template <typename T>
static void land(T* out, const T* dst, size_t n) {
  if (dst != out) memcpy(out, dst, n * sizeof(T));
}

// d = src[0 .. n), copied on `st`
template <typename T>
static int upload_async(DeviceBuf<T>& d, const T* src, size_t n, cudaStream_t st) {
  CU(d.reserve(n));
  if (n) CU(cudaMemcpyAsync(d.get(), src, n * sizeof(T), cudaMemcpyHostToDevice, st));
  return GELATO_OK;
}

// The host-buffer form of a diagnostic with outputs out0 / out1 of bytes0 / bytes1 (NULL: not computed), on lane 0:
// x[n_scen][n_vars] staged and uploaded, launch(x_dev, out0_dev, out1_dev, stream) into the plan's output slots, and
// each output downloaded into the caller's buffer, through the pinned slot when that buffer is pageable.
template <typename Launch>
static int eval_diag(GelatoPlan* p, const double* x, int32_t n_scen, void* out0, size_t bytes0, void* out1, size_t bytes1,
                     Launch launch) {
  CU(cudaSetDevice(p->device));
  int rc = ensure_staging(p, n_scen);
  if (rc) return rc;
  const cudaStream_t st = p->lanes[0].stream;
  const size_t nx = (size_t)n_scen * p->view.n_vars, bytes[2] = {bytes0, bytes1};
  char *const out[2] = {(char*)out0, (char*)out1}, *dst[2];
  for (int k = 0; k < 2; k++)
    if (out[k]) CU(p->d_diag[k].reserve(bytes[k]));
  CU(cudaMemcpyAsync(p->d_x.get(), host_src(x, p->h_x.get(), nx), nx * sizeof(double), cudaMemcpyHostToDevice, st));
  if ((rc = launch(p->d_x.get(), out0 ? p->d_diag[0].get() : nullptr, out1 ? p->d_diag[1].get() : nullptr, st))) return rc;
  for (int k = 0; k < 2; k++) {
    if ((rc = host_dst(out[k], p->h_diag[k], bytes[k], &dst[k]))) return rc;
    if (out[k]) CU(cudaMemcpyAsync(dst[k], p->d_diag[k].get(), bytes[k], cudaMemcpyDeviceToHost, st));
  }
  CU(cudaStreamSynchronize(st));
  for (int k = 0; k < 2; k++) land(out[k], dst[k], bytes[k]);
  return GELATO_OK;
}
}

// The start of replacing a test grid once its lists are built: nothing in flight may still read the grid being
// replaced, then the sections `secs` and the pool of g go to `tg` on lane 0's stream.  The caller uploads its own lists
// on that stream and synchronises it.
static int upload_grid(GelatoPlan* p, TestGrid& tg, const std::vector<MeshSec>& secs, const GelatoMeshGridDesc* g) {
  CU(cudaSetDevice(p->device));
  CU(cudaDeviceSynchronize());
  const int rc = upload_async(tg.sec, secs.data(), secs.size(), p->lanes[0].stream);
  return rc ? rc : upload_async(tg.pool, g->pool, (size_t)g->pool_len, p->lanes[0].stream);
}

static int eval_host(GelatoPlan* p, int which, const double* x, double* out, int32_t n_scen,
                     const int32_t* ids = nullptr) {
  int rc = check_scen(p, n_scen);
  if (rc) return rc;
  if (!x || !out) return fail(GELATO_ERR_ARG, "null buffer");
  CU(cudaSetDevice(p->device));
  if ((rc = ensure_staging(p, n_scen))) return rc;
  const PlanView& v = p->view;
  const Lane& L = p->lanes[0];
  const size_t nx = (size_t)n_scen * v.n_vars;
  const size_t no = (size_t)n_scen * (which == 0 ? (size_t)v.n_rows : (size_t)v.n_vals);
  // a small objfunc call (one NLP, a few scenarios) is launch-latency bound: upload + kernel + download go out as one
  // graph launch through the pinned staging buffers (GELATO_B200_NO_GRAPH=1 keeps the three separate submissions)
  static const bool use_graph = !getenv("GELATO_B200_NO_GRAPH");
  if (which == 0 && !ids && use_graph && (nx + no) * sizeof(double) <= (size_t)64 * 1024) {
    if (p->res_graph && p->res_graph_n != n_scen) drop_graph(p);
    if (!p->res_graph) {
      cudaGraph_t graph = nullptr;
      CU(cudaStreamBeginCapture(L.stream, cudaStreamCaptureModeThreadLocal));
      cudaMemcpyAsync(p->d_x.get(), p->h_x.get(), nx * sizeof(double), cudaMemcpyHostToDevice, L.stream);
      k_residuals<<<(unsigned)p->n_res_blocks * n_scen, GR_THREADS, 0, L.stream>>>(p->view, p->res_blocks, n_scen, nullptr,
                                                                                  p->d_x.get(), p->d_g.get());
      if (p->tab.n_tab > 0)
        k_user_table<<<(unsigned)(((long long)p->tab.n_tab * n_scen * 32 + GT_THREADS - 1) / GT_THREADS), GT_THREADS, 0,
                       L.stream>>>(p->view, p->tab, n_scen, nullptr, p->d_x.get(), nullptr, p->d_g.get());
      cudaMemcpyAsync(p->h_g.get(), p->d_g.get(), no * sizeof(double), cudaMemcpyDeviceToHost, L.stream);
      CU(cudaStreamEndCapture(L.stream, &graph));
      cudaGraphExec_t exec = nullptr;
      cudaError_t ge = cudaGraphInstantiate(&exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ge != cudaSuccess) return fail(GELATO_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ge));
      p->res_graph = GraphExec(exec);
      p->res_graph_n = n_scen;
    }
    memcpy(p->h_x.get(), x, nx * sizeof(double));
    CU(cudaGraphLaunch(p->res_graph, L.stream));
    p->launches++;
    CU(cudaStreamSynchronize(L.stream));
    memcpy(out, p->h_g.get(), no * sizeof(double));
    return GELATO_OK;
  }
  const int32_t* d_ids = nullptr;  // batch slot k evaluates configured scenario ids[k]
  if ((rc = stage_ids(p, ids, n_scen, false, L.stream, &d_ids))) return rc;
  double* d_out = p->d_g.get();
  if (which == 1) {
    if ((rc = ensure_fd_scratch(p, n_scen))) return rc;
    if (!ids) {
      if ((rc = ensure_vals(p, n_scen))) return rc;
      d_out = p->d_vals.get();
    } else {  // constants of each slot's scenario
      CU(p->d_vals_ids.reserve(no));
      d_out = p->d_vals_ids.get();
      for (int k = 0; k < n_scen; k++)
        CU(cudaMemcpyAsync(d_out + (size_t)k * v.n_vals, p->vals_template + (size_t)ids[k] * p->vals_template_sstride,
                           (size_t)v.n_vals * sizeof(double), cudaMemcpyDeviceToDevice, L.stream));
    }
  }
  CU(cudaMemcpyAsync(p->d_x.get(), host_src(x, p->h_x.get(), nx), nx * sizeof(double), cudaMemcpyHostToDevice, L.stream));
  if (which == 0) rc = launch_residuals(p, p->d_x.get(), d_out, n_scen, d_ids, L.stream);
  else rc = launch_jacobian(p, p->d_x.get(), d_out, nullptr, n_scen, L.stream, L, d_ids, false);
  if (rc) return rc;
  double* dst;
  if ((rc = host_dst(out, which == 0 ? p->h_g : p->h_vals, no, &dst))) return rc;
  CU(cudaMemcpyAsync(dst, d_out, no * sizeof(double), cudaMemcpyDeviceToHost, L.stream));
  CU(cudaStreamSynchronize(L.stream));
  land(out, dst, no);
  return GELATO_OK;
}

int gelato_eval_residuals(GelatoPlan* p, const double* x, double* g, int32_t n_scen) {
  return eval_host(p, 0, x, g, n_scen);
}

int gelato_eval_jacobian(GelatoPlan* p, const double* x, double* vals, int32_t n_scen) {
  return eval_host(p, 1, x, vals, n_scen);
}

int gelato_eval_residuals_ids(GelatoPlan* p, const double* x, double* g, int32_t n_scen, const int32_t* scen_ids) {
  if (!scen_ids) return fail(GELATO_ERR_ARG, "null scen_ids");
  return eval_host(p, 0, x, g, n_scen, scen_ids);
}

int gelato_eval_jacobian_ids(GelatoPlan* p, const double* x, double* vals, int32_t n_scen, const int32_t* scen_ids) {
  if (!scen_ids) return fail(GELATO_ERR_ARG, "null scen_ids");
  return eval_host(p, 1, x, vals, n_scen, scen_ids);
}

// ---- mesh error estimate (mesh_error.h) ----
int gelato_plan_set_mesh_grid(GelatoPlan* p, const GelatoMeshGridDesc* g) {
  if (!p || !g || !g->m || !g->off || !g->pool) return fail(GELATO_ERR_ARG, "null argument");
  std::vector<MeshSec> secs;
  std::vector<MeshPt> pts;
  std::vector<MeshInt> ints;
  std::vector<int32_t> int0;
  if (const char* why = build_mesh_grid(g, p->sec_n.data(), p->view.S, secs, pts, ints, int0))
    return fail(GELATO_ERR_ARG, why);
  std::vector<PathPt> path_pts;
  std::vector<int32_t> job0;
  if (const char* why = build_path_points(p->aero_i32.data(), p->view.n_aero, secs, path_pts, job0))
    return fail(GELATO_ERR_ARG, why);
  const cudaStream_t st = p->lanes[0].stream;
  int rc;
  if ((rc = upload_grid(p, p->mesh_grid, secs, g)) || (rc = upload_async(p->d_mesh_pt, pts.data(), pts.size(), st)) ||
      (rc = upload_async(p->d_mesh_int, ints.data(), ints.size(), st)) ||
      (rc = upload_async(p->d_mesh_int0, int0.data(), int0.size(), st)) ||
      (rc = upload_async(p->d_path_pt, path_pts.data(), path_pts.size(), st)) ||
      (rc = upload_async(p->d_path_job0, job0.data(), job0.size(), st)))
    return rc;
  CU(cudaStreamSynchronize(st));
  p->n_mesh_pts = (int)pts.size();
  p->n_mesh_int = (int)ints.size();
  p->mesh_intervals = g->n_int != nullptr;
  p->n_path_pts = (int)path_pts.size();
  return GELATO_OK;
}

// The two launches of one estimate on `st` into err_dev [n_scen][S][11] and / or err_int_dev [n_scen][n_int][11]; the
// point scratch grows to the batch (DeviceBuf::reserve synchronises).
static int launch_mesh_error(GelatoPlan* p, const double* x_dev, double* err_dev, double* err_int_dev, int n_scen,
                             cudaStream_t st) {
  const long long n1 = (long long)n_scen * p->n_mesh_pts, n2 = (long long)n_scen * p->view.S * MESH_STATE;
  if ((std::max(n1, n2) + GM_THREADS - 1) / GM_THREADS > 0x7fffffffLL)
    return fail(GELATO_ERR_ARG, "test points x n_scen exceeds the grid limit");
  CU(p->d_mesh_pts.reserve((size_t)n1 * MESH_PT));
  k_mesh_points<<<(unsigned)((n1 + GM_THREADS - 1) / GM_THREADS), GM_THREADS, 0, st>>>(
      p->view, p->d_mesh_pt.get(), p->mesh_grid.sec.get(), p->mesh_grid.pool.get(), p->n_mesh_pts, n_scen, x_dev, p->d_mesh_pts.get());
  (p->mesh_intervals ? k_mesh_error<true> : k_mesh_error<false>)<<<(unsigned)((n2 + GM_THREADS - 1) / GM_THREADS),
                                                                   GM_THREADS, 0, st>>>(
      p->view, p->mesh_grid.sec.get(), p->d_mesh_int.get(), p->d_mesh_int0.get(), p->mesh_grid.pool.get(), p->n_mesh_pts,
      p->n_mesh_int, n_scen, x_dev, p->d_mesh_pts.get(), err_dev, err_int_dev);
  p->launches += 2;
  CU(cudaGetLastError());
  return GELATO_OK;
}

int gelato_eval_mesh_error_dev(GelatoPlan* p, const double* x_dev, double* err_dev, int32_t n_scen, void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  if (!p->n_mesh_pts) return fail(GELATO_ERR_ARG, GELATO_NO_MESH_GRID);
  if (!x_dev || !err_dev) return fail(GELATO_ERR_ARG, "null buffer");
  return launch_mesh_error(p, x_dev, err_dev, nullptr, n_scen, st);
}

int gelato_eval_mesh_error(GelatoPlan* p, const double* x, double* err, int32_t n_scen) {
  int rc = check_scen(p, n_scen);
  if (rc) return rc;
  if (!p->n_mesh_pts) return fail(GELATO_ERR_ARG, GELATO_NO_MESH_GRID);
  if (!x || !err) return fail(GELATO_ERR_ARG, "null buffer");
  const size_t ne = (size_t)n_scen * p->view.S * MESH_STATE;
  return eval_diag(p, x, n_scen, err, ne * sizeof(double), nullptr, 0,
                   [&](const double* xd, void* o0, void*, cudaStream_t st) {
                     return launch_mesh_error(p, xd, (double*)o0, nullptr, n_scen, st);
                   });
}

int gelato_eval_mesh_error_intervals_dev(GelatoPlan* p, const double* x_dev, double* err_int_dev, int32_t n_scen,
                                         void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  if (!p->n_mesh_pts) return fail(GELATO_ERR_ARG, GELATO_NO_MESH_GRID);
  if (!x_dev || !err_int_dev) return fail(GELATO_ERR_ARG, "null buffer");
  return launch_mesh_error(p, x_dev, nullptr, err_int_dev, n_scen, st);
}

int gelato_eval_mesh_error_intervals(GelatoPlan* p, const double* x, double* err_int, int32_t n_scen) {
  int rc = check_scen(p, n_scen);
  if (rc) return rc;
  if (!p->n_mesh_pts) return fail(GELATO_ERR_ARG, GELATO_NO_MESH_GRID);
  if (!x || !err_int) return fail(GELATO_ERR_ARG, "null buffer");
  const size_t ne = (size_t)n_scen * p->n_mesh_int * MESH_STATE;
  return eval_diag(p, x, n_scen, err_int, ne * sizeof(double), nullptr, 0,
                   [&](const double* xd, void* o0, void*, cudaStream_t st) {
                     return launch_mesh_error(p, xd, nullptr, (double*)o0, n_scen, st);
                   });
}

// ---- path check (mesh_error.h) ----
// The launches of one check on `st`: none without aero jobs, k_path_points only when a job runs over a whole section;
// the point scratch grows to the batch (DeviceBuf::reserve synchronises).
static int launch_path_check(GelatoPlan* p, const double* x_dev, double* res_dev, int32_t* at_dev, int n_scen,
                             cudaStream_t st) {
  const int n_aero = p->view.n_aero, n_pts = p->n_path_pts;
  if (!n_aero) return GELATO_OK;
  const long long n1 = (long long)n_scen * n_pts, n2 = (long long)n_scen * n_aero;
  if ((std::max(n1, n2) + GM_THREADS - 1) / GM_THREADS > 0x7fffffffLL)
    return fail(GELATO_ERR_ARG, "test points x n_scen exceeds the grid limit");
  CU(p->d_path_r.reserve((size_t)n1));
  if (n1 > 0) {
    k_path_points<<<(unsigned)((n1 + GM_THREADS - 1) / GM_THREADS), GM_THREADS, 0, st>>>(
        p->view, p->d_path_pt.get(), p->mesh_grid.sec.get(), p->mesh_grid.pool.get(), n_pts, n_scen, x_dev, p->d_path_r.get());
    p->launches++;
  }
  k_path_min<<<(unsigned)((n2 + GM_THREADS - 1) / GM_THREADS), GM_THREADS, 0, st>>>(
      n_aero, p->d_path_job0.get(), n_pts, n_scen, p->d_path_r.get(), res_dev, at_dev);
  p->launches++;
  CU(cudaGetLastError());
  return GELATO_OK;
}

int gelato_eval_path_check_dev(GelatoPlan* p, const double* x_dev, double* res_dev, int32_t* at_dev, int32_t n_scen,
                               void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  if (!p->n_mesh_pts) return fail(GELATO_ERR_ARG, GELATO_NO_MESH_GRID);
  if (!x_dev || (p->view.n_aero && (!res_dev || !at_dev))) return fail(GELATO_ERR_ARG, "null buffer");
  return launch_path_check(p, x_dev, res_dev, at_dev, n_scen, st);
}

int gelato_eval_path_check(GelatoPlan* p, const double* x, double* res, int32_t* at, int32_t n_scen) {
  int rc = check_scen(p, n_scen);
  if (rc) return rc;
  if (!p->n_mesh_pts) return fail(GELATO_ERR_ARG, GELATO_NO_MESH_GRID);
  if (!x || (p->view.n_aero && (!res || !at))) return fail(GELATO_ERR_ARG, "null buffer");
  if (!p->view.n_aero) return GELATO_OK;
  const size_t na = (size_t)n_scen * p->view.n_aero;
  return eval_diag(p, x, n_scen, res, na * sizeof(double), at, na * sizeof(int32_t),
                   [&](const double* xd, void* o0, void* o1, cudaStream_t st) {
                     return launch_path_check(p, xd, (double*)o0, (int32_t*)o1, n_scen, st);
                   });
}

// ---- path rows (mesh_error.h) ----
int gelato_plan_set_path_rows(GelatoPlan* p, const GelatoMeshGridDesc* g) {
  if (!p || !g || !g->m || !g->off || !g->pool) return fail(GELATO_ERR_ARG, "null argument");
  std::vector<MeshSec> secs;
  std::vector<MeshPt> pts;
  if (const char* why = build_mesh_grid(g, p->sec_n.data(), p->view.S, secs, pts)) return fail(GELATO_ERR_ARG, why);
  std::vector<PathRow> rows;
  long long n_vals = 0;
  if (const char* why = build_path_rows(p->aero_i32.data(), p->view.n_aero, p->sec_n.data(), secs, g->pool, rows, &n_vals))
    return fail(GELATO_ERR_ARG, why);
  const cudaStream_t st = p->lanes[0].stream;
  int rc;
  if ((rc = upload_grid(p, p->prow_grid, secs, g)) || (rc = upload_async(p->d_prow, rows.data(), rows.size(), st)))
    return rc;
  CU(cudaStreamSynchronize(st));
  p->prow.swap(rows);
  p->prow_vals = n_vals;
  p->prow_set = true;
  return GELATO_OK;
}

int gelato_plan_path_rows(const GelatoPlan* p, int32_t* n_rows, int64_t* n_vals, int32_t* job, int32_t* l, int64_t* off) {
  if (!p || !n_rows || !n_vals) return fail(GELATO_ERR_ARG, "null argument");
  if (!p->prow_set) return fail(GELATO_ERR_ARG, GELATO_NO_PATH_ROWS);
  *n_rows = (int32_t)p->prow.size();
  *n_vals = p->prow_vals;
  for (size_t k = 0; k < p->prow.size(); k++) {
    if (job) job[k] = p->prow[k].job;
    if (l) l[k] = p->prow[k].l;
    if (off)
      for (int c = 0; c < PR_OFFS; c++) off[k * PR_OFFS + c] = p->prow[k].off[c];
  }
  return GELATO_OK;
}

// The launch of one evaluation on `st` in the plan's finite-difference mode: PATH_LANES threads per row with a Jacobian,
// one without.  Nothing without rows or outputs.
static int launch_path_rows(GelatoPlan* p, const double* x_dev, double* g_dev, double* vals_dev, int n_scen, cudaStream_t st) {
  const int n_rows = (int)p->prow.size();
  if (!n_rows || (!g_dev && !vals_dev)) return GELATO_OK;
  const int lanes = vals_dev ? PATH_LANES : 1;
  const long long nt = (long long)n_scen * n_rows * lanes;
  if ((nt + GP_THREADS - 1) / GP_THREADS > 0x7fffffffLL) return fail(GELATO_ERR_ARG, "path rows x n_scen exceeds the grid limit");
  const int central = p->fd_mode == GELATO_FD_CENTRAL;
  k_path_rows<<<(unsigned)((nt + GP_THREADS - 1) / GP_THREADS), GP_THREADS, 0, st>>>(
      p->view, p->d_prow.get(), p->prow_grid.sec.get(), p->prow_grid.pool.get(), n_rows, p->prow_vals, n_scen, lanes, central,
      central ? p->fd_step : p->view.un.dx, x_dev, g_dev, vals_dev);
  p->launches++;
  CU(cudaGetLastError());
  return GELATO_OK;
}

int gelato_eval_path_rows_dev(GelatoPlan* p, const double* x_dev, double* g_dev, double* vals_dev, int32_t n_scen,
                              void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  if (!p->prow_set) return fail(GELATO_ERR_ARG, GELATO_NO_PATH_ROWS);
  if (!x_dev) return fail(GELATO_ERR_ARG, "null buffer");
  return launch_path_rows(p, x_dev, g_dev, vals_dev, n_scen, st);
}

int gelato_eval_path_rows(GelatoPlan* p, const double* x, double* g_path, double* vals_path, int32_t n_scen) {
  int rc = check_scen(p, n_scen);
  if (rc) return rc;
  if (!p->prow_set) return fail(GELATO_ERR_ARG, GELATO_NO_PATH_ROWS);
  if (!x) return fail(GELATO_ERR_ARG, "null buffer");
  if (p->prow.empty() || (!g_path && !vals_path)) return GELATO_OK;
  const size_t ng = (size_t)n_scen * p->prow.size(), nv = (size_t)n_scen * (size_t)p->prow_vals;
  return eval_diag(p, x, n_scen, g_path, ng * sizeof(double), vals_path, nv * sizeof(double),
                   [&](const double* xd, void* o0, void* o1, cudaStream_t st) {
                     return launch_path_rows(p, xd, (double*)o0, (double*)o1, n_scen, st);
                   });
}

int gelato_pack_xdep_dev(GelatoPlan* p, const double* vals_dev, double* packed_dev, int32_t n_scen, void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  if (!p->d_xdep) return fail(GELATO_ERR_ARG, "the plan was created without xdep_idx");
  if (n_scen > 65535) return fail(GELATO_ERR_ARG, "n_scen > 65535 in update mode (gridDim.y)");
  const int threads = 256;
  const int bx = (int)std::min<long long>((p->n_xdep + threads - 1) / threads, 4096);
  k_pack_xdep<<<dim3(bx, n_scen), threads, 0, st>>>(vals_dev, p->d_xdep, p->n_xdep, p->view.n_vals, packed_dev);
  p->launches++;
  CU(cudaGetLastError());
  return GELATO_OK;
}

int gelato_jacobian_template(GelatoPlan* p, double* vals, int32_t n_scen) {
  int rc = check_scen(p, n_scen);
  if (rc) return rc;
  if (!vals) return fail(GELATO_ERR_ARG, "null buffer");
  CU(cudaSetDevice(p->device));
  const size_t nv = (size_t)p->view.n_vals;
  if (p->vals_template_sstride) {
    CU(cudaMemcpy(vals, p->vals_template, (size_t)n_scen * nv * sizeof(double), cudaMemcpyDeviceToHost));
  } else {
    CU(cudaMemcpy(vals, p->vals_template, nv * sizeof(double), cudaMemcpyDeviceToHost));
    for (int s = 1; s < n_scen; s++) memcpy(vals + (size_t)s * nv, vals, nv * sizeof(double));
  }
  return GELATO_OK;
}

int gelato_set_update_zero_copy(GelatoPlan* p, int32_t on) {
  if (!p) return fail(GELATO_ERR_ARG, "null plan");
  p->update_zero_copy = on ? 1 : 0;
  return GELATO_OK;
}

int gelato_set_host_threads(GelatoPlan* p, int32_t n) {
  if (!p || n < 0) return fail(GELATO_ERR_ARG, "bad thread count");
  p->host_threads = n;
  return GELATO_OK;
}

using gelato_host::scatter_parallel;

// The slices a host-buffer call cuts its batch into, each on a lane of its own (measured: profiles/r01v_e2e.txt).
struct Slices {
  int n_scen, n;
  int lo(int k) const { return (int)((long long)n_scen * k / n); }
};
static Slices slices_for(const GelatoPlan* p, int n_scen) {
  const int n = p->update_slices > 0 ? p->update_slices : n_scen / 16;
  return Slices{n_scen, std::max(1, std::min(n, std::min(n_scen, 8)))};
}

// lanes [0, n), each with n_chunks chunk events
static int ensure_lanes(GelatoPlan* p, int n, int n_chunks) {
  int rc;
  while ((int)p->lanes.size() < n)
    if ((rc = add_lane(p))) return rc;
  for (int k = 0; k < n; k++)
    while ((int)p->lanes[k].chunk_ev.size() < n_chunks) {
      p->lanes[k].chunk_ev.emplace_back();
      CU(cudaEventCreateWithFlags(p->lanes[k].chunk_ev.back().out(), cudaEventDisableTiming));
    }
  return GELATO_OK;
}

// Slice k of a batch on lane k: after slice k-1's upload (uploads go one after the other), the slice's x goes up from
// hx and one Jacobian evaluation of its scenarios writes out_dev (and g_dev), both offset to the slice already.
static int launch_slice(GelatoPlan* p, const Slices& sl, int k, const double* hx, double* out_dev, double* g_dev,
                        const int32_t* ids, bool packed) {
  const Lane& L = p->lanes[k];
  const int s0 = sl.lo(k), ns = sl.lo(k + 1) - s0;
  const size_t nx = (size_t)p->view.n_vars;
  double* const dx = p->d_x.get() + (size_t)s0 * nx;
  if (k > 0) CU(cudaStreamWaitEvent(L.stream, p->lanes[k - 1].ev_h2d, 0));
  CU(cudaMemcpyAsync(dx, hx + (size_t)s0 * nx, (size_t)ns * nx * sizeof(double), cudaMemcpyHostToDevice, L.stream));
  CU(cudaEventRecord(L.ev_h2d, L.stream));
  return launch_jacobian(p, dx, out_dev, g_dev, ns, L.stream, L, ids ? ids + s0 : nullptr, packed, s0);
}

// shared body of gelato_eval_jacobian_update / gelato_eval_pair_update; g == NULL: Jacobian only.
// The batch is cut into slices of scenarios, each on its own lane of streams: slice k's upload and kernels
// overlap slice k-1's device->host traffic (PCIe is full duplex), and the host threads scatter slice k-1's
// packed slots meanwhile.  Per slice: upload x -> { residual kernel -> copy g | Jacobian kernel -> transfers }.
static int eval_update(GelatoPlan* p, const double* x, double* g, double* vals, int32_t n_scen) {
  int rc = check_scen(p, n_scen);
  if (rc) return rc;
  if (!x || !vals) return fail(GELATO_ERR_ARG, "null buffer");
  if (!p->d_xdep) return fail(GELATO_ERR_ARG, "the plan was created without xdep_idx");
  if (n_scen > 65535) return fail(GELATO_ERR_ARG, "n_scen > 65535 in update mode (gridDim.y)");
  CU(cudaSetDevice(p->device));
  if ((rc = ensure_staging(p, n_scen))) return rc;
  if ((rc = ensure_vals(p, n_scen))) return rc;
  if ((rc = ensure_fd_scratch(p, n_scen))) return rc;
  const PlanView& v = p->view;
  CU(p->d_pack.reserve((size_t)n_scen * p->n_xdep));
  CU(p->h_pack.reserve((size_t)n_scen * p->n_xdep));
  const double* hx = host_src(x, p->h_x.get(), (size_t)n_scen * v.n_vars);
  const size_t nv = (size_t)n_scen * (size_t)v.n_vals, ng = (size_t)n_scen * v.n_rows;
  double* g_dst;
  if ((rc = host_dst(g, p->h_g, ng, &g_dst))) return rc;
  // A small Jacobian (one NLP of a few hundred nodes) is cheaper to bring down whole than through the gather / strided
  // copies / host scatter below: the staging copy on the device always holds the complete value vector (constants
  // filled once, x-dependent slots rewritten by every launch), so one contiguous copy refreshes the caller's buffer
  // to the same bits.
  if (nv * sizeof(double) <= (size_t)512 * 1024) {
    const Lane& L = p->lanes[0];
    CU(cudaMemcpyAsync(p->d_x.get(), hx, (size_t)n_scen * v.n_vars * sizeof(double), cudaMemcpyHostToDevice, L.stream));
    if ((rc = launch_jacobian(p, p->d_x.get(), p->d_vals.get(), g ? p->d_g.get() : nullptr, n_scen, L.stream, L, nullptr,
                              false)))
      return rc;
    double* v_dst;
    if ((rc = host_dst(vals, p->h_vals, nv, &v_dst))) return rc;
    CU(cudaMemcpyAsync(v_dst, p->d_vals.get(), nv * sizeof(double), cudaMemcpyDeviceToHost, L.stream));
    if (g) CU(cudaMemcpyAsync(g_dst, p->d_g.get(), ng * sizeof(double), cudaMemcpyDeviceToHost, L.stream));
    CU(cudaStreamSynchronize(L.stream));
    land(vals, v_dst, nv);
    if (g) land(g, g_dst, ng);
    return GELATO_OK;
  }

  // Which slots travel packed (gathered on the device, copied, scattered by the host pool) and which go
  // straight to their place: a page-locked `vals` takes the long runs of consecutive slots through the copy
  // engine (one strided 2-D copy per run covers a slice's scenarios) and, in zero-copy mode, the scattered
  // rest through a kernel that stores into the buffer's device mapping.
  const bool direct = is_pinned(vals);
  const int64_t* pack_idx_dev = direct ? p->d_xdep_small : p->d_xdep;
  const int64_t* pack_idx_host = direct ? p->h_small.data() : p->h_xdep.data();
  long long n_pack = direct ? p->n_small : p->n_xdep;
  double* dev_view = nullptr;  // the device's address of the caller's page-locked buffer
  if (direct && p->update_zero_copy && n_pack > 0) {
    if (cudaHostGetDevicePointer((void**)&dev_view, vals, 0) != cudaSuccess) {
      cudaGetLastError();  // registered without a device mapping: the scattered slots travel packed instead
      dev_view = nullptr;
    }
  }
  const bool zero_copy = dev_view != nullptr;

  int threads = p->host_threads > 0 ? p->host_threads : (int)std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
  if ((long long)n_scen * n_pack < (1LL << 18)) threads = 1;
  threads = std::min(threads, (int)n_scen);
  const Slices sl = slices_for(p, n_scen);
  // one slice: the packed slots come down in chunks so the scatter of chunk k overlaps the copy of chunk k+1
  const int n_chunks = (sl.n == 1 && n_scen >= 4 * threads && threads > 1) ? 4 : 1;
  if ((rc = ensure_lanes(p, sl.n, n_chunks))) return rc;
  const int32_t* ids;  // the slices' scenario parameter blocks
  if ((rc = stage_ids(p, nullptr, n_scen, sl.n > 1, p->lanes[0].stream, &ids))) return rc;
  auto chunk_lo = [&](int k, int c) {
    const int s0 = sl.lo(k), s1 = sl.lo(k + 1);
    return s0 + (int)((long long)(s1 - s0) * c / n_chunks);
  };

  for (int k = 0; k < sl.n; k++) {
    const Lane& L = p->lanes[k];
    const int s0 = sl.lo(k), ns = sl.lo(k + 1) - s0;
    double* const dg = p->d_g.get() + (size_t)s0 * v.n_rows;
    double* const dvals = p->d_vals.get() + (size_t)s0 * v.n_vals;
    double* const hvals = vals + (size_t)s0 * v.n_vals;
    // g != NULL: pair evaluation, the residual rows come out of the same launches
    if ((rc = launch_slice(p, sl, k, hx, dvals, g ? dg : nullptr, ids, false))) return rc;
    if (g) {  // its copy travels on the side stream, next to the Jacobian's transfers
      CU(cudaEventRecord(L.ev_g, L.stream));
      CU(cudaStreamWaitEvent(L.pair_stream, L.ev_g, 0));
      CU(cudaMemcpyAsync(g_dst + (size_t)s0 * v.n_rows, dg, (size_t)ns * v.n_rows * sizeof(double), cudaMemcpyDeviceToHost,
                         L.pair_stream));
      CU(cudaEventRecord(L.ev_gdone, L.pair_stream));
    }

    // the long runs, on the lane's copy stream once `after` has happened
    auto issue_runs = [&](cudaEvent_t after) -> int {
      CU(cudaStreamWaitEvent(L.copy_stream, after, 0));
      const size_t pitch = (size_t)v.n_vals * sizeof(double);
      for (const auto& run : p->big_runs)
        CU(cudaMemcpy2DAsync(hvals + run.first, pitch, dvals + run.first, pitch, (size_t)run.second * sizeof(double),
                             (size_t)ns, cudaMemcpyDeviceToHost, L.copy_stream));
      CU(cudaEventRecord(L.ev_copy, L.copy_stream));
      return GELATO_OK;
    };
    const int gpu_threads = 256;
    const int bx = (int)std::max<long long>(1, std::min<long long>((n_pack + gpu_threads - 1) / gpu_threads, 4096));
    if (direct && (zero_copy || n_pack == 0)) {
      CU(cudaEventRecord(L.ev_kernel, L.stream));
      if (zero_copy) {
        k_scatter_xdep_host<<<dim3(bx, ns), gpu_threads, 0, L.stream>>>(dvals, pack_idx_dev, n_pack, v.n_vals,
                                                                       dev_view + (size_t)s0 * v.n_vals);
        p->launches++;
        CU(cudaGetLastError());
      }
      if ((rc = issue_runs(L.ev_kernel))) return rc;
    } else if (n_pack > 0) {
      k_pack_xdep<<<dim3(bx, ns), gpu_threads, 0, L.stream>>>(dvals, pack_idx_dev, n_pack, v.n_vals,
                                                             p->d_pack.get() + (size_t)s0 * n_pack);
      p->launches++;
      CU(cudaGetLastError());
      for (int c = 0; c < n_chunks; c++) {
        const size_t off = (size_t)chunk_lo(k, c) * n_pack, cnt = (size_t)(chunk_lo(k, c + 1) - chunk_lo(k, c)) * n_pack;
        CU(cudaMemcpyAsync(p->h_pack.get() + off, p->d_pack.get() + off, cnt * sizeof(double), cudaMemcpyDeviceToHost,
                           L.stream));
        CU(cudaEventRecord(L.chunk_ev[c], L.stream));
      }
      // the packed slots cross PCIe first: the host threads scatter them while the long runs follow
      if (direct && (rc = issue_runs(L.chunk_ev[n_chunks - 1]))) return rc;
    }
  }
  if (!zero_copy && n_pack > 0)
    for (int k = 0; k < sl.n; k++)
      for (int c = 0; c < n_chunks; c++) {
        CU(cudaEventSynchronize(p->lanes[k].chunk_ev[c]));
        scatter_parallel(pack_idx_host, n_pack, p->h_pack.get(), vals, v.n_vals, chunk_lo(k, c), chunk_lo(k, c + 1), threads);
      }
  for (int k = 0; k < sl.n; k++) {
    const Lane& L = p->lanes[k];
    if (direct) CU(cudaStreamWaitEvent(L.stream, L.ev_copy, 0));
    if (g) CU(cudaStreamWaitEvent(L.stream, L.ev_gdone, 0));
    CU(cudaStreamSynchronize(L.stream));
  }
  if (g) land(g, g_dst, ng);
  return GELATO_OK;
}

// Packed host entry points: x[n_scen][n_vars] up, the pair (or Jacobian-only) evaluation, then g[n_scen][n_rows] and
// packed[n_scen][n_pack] down as CONTIGUOUS copies -- no gather kernel, no host scatter.  Pipelined over slices of
// the batch like update mode: slice k's upload and kernels overlap slice k-1's device->host copies (PCIe is full
// duplex).  Page-locked caller buffers (gelato_host_alloc) are DMA'd directly, others staged.
static int eval_packed(GelatoPlan* p, const double* x, double* g, double* packed, int32_t n_scen, const int32_t* scen_ids) {
  int rc = check_scen(p, n_scen);
  if (rc) return rc;
  if (!x || !packed) return fail(GELATO_ERR_ARG, "null buffer");
  const PlanView& v = p->view;
  CU(cudaSetDevice(p->device));
  if ((rc = ensure_staging(p, n_scen))) return rc;
  if ((rc = ensure_fd_scratch(p, n_scen))) return rc;
  const size_t np = (size_t)p->n_pack;
  CU(p->d_packed.reserve((size_t)n_scen * np));
  const Slices sl = slices_for(p, n_scen);
  if ((rc = ensure_lanes(p, sl.n, 0))) return rc;
  // scenario ids of the batch slots: the caller's subset, or 0, 1, 2 ... when the batch is cut into slices; the first
  // upload waits for them
  const int32_t* ids;
  if ((rc = stage_ids(p, scen_ids, n_scen, sl.n > 1, p->lanes[0].stream, &ids))) return rc;
  const double* hx = host_src(x, p->h_x.get(), (size_t)n_scen * v.n_vars);
  double *g_dst, *pk_dst;
  if ((rc = host_dst(g, p->h_g, (size_t)n_scen * v.n_rows, &g_dst))) return rc;
  if ((rc = host_dst(packed, p->h_packed, (size_t)n_scen * np, &pk_dst))) return rc;
  for (int k = 0; k < sl.n; k++) {
    const Lane& L = p->lanes[k];
    const int s0 = sl.lo(k), ns = sl.lo(k + 1) - s0;
    double* const dg = p->d_g.get() + (size_t)s0 * v.n_rows;
    double* const dpk = p->d_packed.get() + (size_t)s0 * np;
    if ((rc = launch_slice(p, sl, k, hx, dpk, g ? dg : nullptr, ids, true))) return rc;
    // both results on the lane's copy stream, after everything of the slice has been computed
    CU(cudaEventRecord(L.ev_kernel, L.stream));
    CU(cudaStreamWaitEvent(L.copy_stream, L.ev_kernel, 0));
    if (g)
      CU(cudaMemcpyAsync(g_dst + (size_t)s0 * v.n_rows, dg, (size_t)ns * v.n_rows * sizeof(double), cudaMemcpyDeviceToHost,
                         L.copy_stream));
    CU(cudaMemcpyAsync(pk_dst + (size_t)s0 * np, dpk, (size_t)ns * np * sizeof(double), cudaMemcpyDeviceToHost, L.copy_stream));
    CU(cudaEventRecord(L.ev_copy, L.copy_stream));
  }
  for (int k = 0; k < sl.n; k++) CU(cudaEventSynchronize(p->lanes[k].ev_copy));
  if (g) land(g, g_dst, (size_t)n_scen * v.n_rows);
  land(packed, pk_dst, (size_t)n_scen * np);
  return GELATO_OK;
}

int gelato_eval_pair_packed(GelatoPlan* p, const double* x, double* g, double* packed, int32_t n_scen) {
  if (!g) return fail(GELATO_ERR_ARG, "null buffer");
  return eval_packed(p, x, g, packed, n_scen, nullptr);
}

int gelato_eval_jacobian_packed(GelatoPlan* p, const double* x, double* packed, int32_t n_scen) {
  return eval_packed(p, x, nullptr, packed, n_scen, nullptr);
}

int gelato_eval_pair_packed_ids(GelatoPlan* p, const double* x, double* g, double* packed, int32_t n_scen,
                                const int32_t* scen_ids) {
  if (!g || !scen_ids) return fail(GELATO_ERR_ARG, "null buffer");
  return eval_packed(p, x, g, packed, n_scen, scen_ids);
}

int64_t gelato_plan_n_pack(const GelatoPlan* p) { return p ? p->n_pack : 0; }

int gelato_plan_packed_map(const GelatoPlan* p, int64_t* full_slot, int64_t* src, double* sgn) {
  if (!p || !full_slot || !src || !sgn) return fail(GELATO_ERR_ARG, "null argument");
  std::copy(p->pk_full.begin(), p->pk_full.end(), full_slot);
  std::copy(p->pk_src.begin(), p->pk_src.end(), src);
  std::copy(p->pk_sgn.begin(), p->pk_sgn.end(), sgn);
  return GELATO_OK;
}

int gelato_set_update_slices(GelatoPlan* p, int32_t n) {
  if (!p || n < 0) return fail(GELATO_ERR_ARG, "bad slice count");
  p->update_slices = n;
  return GELATO_OK;
}

int gelato_eval_jacobian_update(GelatoPlan* p, const double* x, double* vals, int32_t n_scen) {
  return eval_update(p, x, nullptr, vals, n_scen);
}

int gelato_eval_pair_update(GelatoPlan* p, const double* x, double* g, double* vals, int32_t n_scen) {
  if (!g) return fail(GELATO_ERR_ARG, "null buffer");
  return eval_update(p, x, g, vals, n_scen);
}

// Measurement only: device times (ms) of the transfer pieces of update mode, each alone, for a page-locked
// `vals` after a gelato_eval_*_update call: [0] the 2-D copies of the long runs, [1] the zero-copy kernel of the
// scattered slots, [2] both at once, [3] pack kernel + one contiguous copy of the scattered slots (no host
// scatter), [4] one contiguous copy of as many bytes as all x-dependent slots, [5] the residual copy.
int gelato_probe_update(GelatoPlan* p, double* vals, int32_t n_scen, int reps, float* out_ms) {
  int rc = check_scen(p, n_scen);
  if (rc) return rc;
  if (!vals || !out_ms || reps <= 0 || !is_pinned(vals)) return fail(GELATO_ERR_ARG, "page-locked vals required");
  if (!p->d_xdep || (size_t)n_scen * p->n_xdep > p->d_pack.size())
    return fail(GELATO_ERR_ARG, "call gelato_eval_jacobian_update first");
  const PlanView& v = p->view;
  const Lane& L = p->lanes[0];
  double* dev_view = nullptr;
  CU(cudaHostGetDevicePointer((void**)&dev_view, vals, 0));
  const size_t pitch = (size_t)v.n_vals * sizeof(double);
  const int threads = 256;
  const int bx = (int)std::min<long long>((p->n_small + threads - 1) / threads, 4096);
  auto copies = [&]() {
    for (const auto& run : p->big_runs)
      cudaMemcpy2DAsync(vals + run.first, pitch, p->d_vals.get() + run.first, pitch, (size_t)run.second * sizeof(double),
                        (size_t)n_scen, cudaMemcpyDeviceToHost, L.copy_stream);
  };
  auto zero_copy = [&]() {
    if (p->n_small > 0)
      k_scatter_xdep_host<<<dim3(bx, n_scen), threads, 0, L.stream>>>(p->d_vals.get(), p->d_xdep_small, p->n_small, v.n_vals,
                                                                       dev_view);
  };
  for (int piece = 0; piece < 6; piece++) {
    CU(cudaDeviceSynchronize());
    CU(cudaEventRecord(p->ev0, L.stream));
    CU(cudaStreamWaitEvent(L.copy_stream, p->ev0, 0));
    for (int r = 0; r < reps; r++) {
      if (piece == 0 || piece == 2) copies();
      if (piece == 1 || piece == 2) zero_copy();
      if (piece == 3 && p->n_small > 0) {
        k_pack_xdep<<<dim3(bx, n_scen), threads, 0, L.stream>>>(p->d_vals.get(), p->d_xdep_small, p->n_small, v.n_vals,
                                                               p->d_pack.get());
        cudaMemcpyAsync(p->h_pack.get(), p->d_pack.get(), (size_t)n_scen * p->n_small * sizeof(double), cudaMemcpyDeviceToHost,
                        L.stream);
      }
      if (piece == 4)
        cudaMemcpyAsync(p->h_pack.get(), p->d_pack.get(), (size_t)n_scen * p->n_xdep * sizeof(double), cudaMemcpyDeviceToHost,
                        L.stream);
      if (piece == 5)
        cudaMemcpyAsync(p->h_g.get(), p->d_g.get(), (size_t)n_scen * v.n_rows * sizeof(double), cudaMemcpyDeviceToHost, L.stream);
    }
    CU(cudaEventRecord(L.ev_copy, L.copy_stream));
    CU(cudaStreamWaitEvent(L.stream, L.ev_copy, 0));
    CU(cudaEventRecord(p->ev1, L.stream));
    CU(cudaEventSynchronize(p->ev1));
    CU(cudaGetLastError());
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
    out_ms[piece] = ms / reps;
  }
  return GELATO_OK;
}

int gelato_host_alloc(size_t bytes, void** out) {
  if (!out) return fail(GELATO_ERR_ARG, "null");
  CU(cudaMallocHost(out, bytes));
  return GELATO_OK;
}

int gelato_host_free(void* ptr) {
  if (ptr) CU(cudaFreeHost(ptr));
  return GELATO_OK;
}

// Measurement helper: enqueue exactly ONE kernel on `stream` (0 residual kernel | 2 heavy Jacobian kernel |
// 3 light Jacobian kernel | 4 the residual kernel's non-dynamics blocks; out_dev = g for 0 and 4), COO or packed
// output, g_dev != NULL: with the pair evaluation's defect rows -- so that a benchmark can bracket it with its own
// CUDA events.
int gelato_launch_kernel_dev(GelatoPlan* p, int which, const double* x_dev, double* out_dev, double* g_dev, int32_t n_scen,
                             int32_t packed, void* stream) {
  cudaStream_t st;
  int rc = begin_dev(p, n_scen, stream, &st);
  if (rc) return rc;
  PlanView v = p->view;
  v.packed = packed ? 1 : 0;
  if (which == 0) {
    k_residuals<<<(unsigned)p->n_res_blocks * n_scen, GR_THREADS, 0, st>>>(v, p->res_blocks, n_scen, nullptr, x_dev, out_dev);
  } else if (which == 1) {
    return launch_jacobian_pass(p, p->view.un.dx, x_dev, out_dev, g_dev, n_scen, st, p->lanes[0], nullptr, packed != 0);
  } else if (which == 2) {
    if (p->n_jac_heavy == 0) return fail(GELATO_ERR_ARG, "the plan has no heavy blocks");
    k_jacobian_heavy<<<(unsigned)p->n_jac_heavy * n_scen, GJ_THREADS, 0, st>>>(v, p->jac_heavy, n_scen, nullptr, x_dev, out_dev, g_dev);
  } else if (which == 3) {
    if (p->n_jac_light == 0) return fail(GELATO_ERR_ARG, "the plan has no light blocks");
    k_jacobian_light<<<(unsigned)p->n_jac_light * n_scen, GJ_THREADS, 0, st>>>(v, p->jac_light, n_scen, nullptr, x_dev, out_dev, g_dev);
  } else if (which == 5) {
    if (p->n_vac == 0) return fail(GELATO_ERR_ARG, "the plan has no vacuum nodes");
    const int per = (p->n_vac + 31) / 32;
    k_jacobian_noair<<<(unsigned)per * n_scen, GV_THREADS, 0, st>>>(v, p->vac_first, p->n_vac, n_scen, nullptr, x_dev, out_dev, g_dev);
  } else if (which == 6) {  // the block kernel alone, as an evaluation launches it
    const int nb = g_dev ? p->n_jac_blocks : p->n_jac_main;
    if (nb == 0) return fail(GELATO_ERR_ARG, "the plan has no Jacobian blocks");
    k_jacobian<<<(unsigned)nb * n_scen, GJ_THREADS, 0, st>>>(v, p->jac_blocks, n_scen, nullptr, x_dev, out_dev, g_dev);
  } else {
    return fail(GELATO_ERR_ARG, "which must be 0, 1, 2, 3, 5 or 6");
  }
  p->launches++;
  CU(cudaGetLastError());
  return GELATO_OK;
}

int gelato_time_kernel(GelatoPlan* p, int which, const double* x_dev, double* out_dev, int32_t n_scen, int reps,
                       float* avg_ms) {
  int rc = check_scen(p, n_scen);
  if (rc) return rc;
  if (reps <= 0 || !avg_ms) return fail(GELATO_ERR_ARG, "bad reps");
  CU(cudaSetDevice(p->device));
  const Lane& L = p->lanes[0];
  CU(cudaStreamSynchronize(L.stream));
  CU(cudaEventRecord(p->ev0, L.stream));
  for (int i = 0; i < reps; i++) {
    if (which == 0) {
      k_residuals<<<(unsigned)p->n_res_blocks * n_scen, GR_THREADS, 0, L.stream>>>(p->view, p->res_blocks, n_scen, nullptr, x_dev, out_dev);
    } else if (which == 1) {  // the whole Jacobian evaluation (heavy and light kernels)
      if ((rc = launch_jacobian_pass(p, p->view.un.dx, x_dev, out_dev, nullptr, n_scen, L.stream, L, nullptr, false)))
        return rc;
      continue;
    } else if (which == 2) {  // the heavy roles' blocks alone (air dynamics + aero rows)
      if (p->n_jac_heavy > 0)
        k_jacobian_heavy<<<(unsigned)p->n_jac_heavy * n_scen, GJ_THREADS, 0, L.stream>>>(p->view, p->jac_heavy, n_scen, nullptr,
                                                                                        x_dev, out_dev, nullptr);
    } else {  // the light roles' blocks alone
      if (p->n_jac_light > 0)
        k_jacobian_light<<<(unsigned)p->n_jac_light * n_scen, GJ_THREADS, 0, L.stream>>>(p->view, p->jac_light, n_scen, nullptr,
                                                                                        x_dev, out_dev, nullptr);
    }
    p->launches++;
  }
  CU(cudaEventRecord(p->ev1, L.stream));
  CU(cudaEventSynchronize(p->ev1));
  CU(cudaGetLastError());
  float ms = 0.f;
  CU(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
  *avg_ms = ms / reps;
  return GELATO_OK;
}

int gelato_selftest_unfused(int device, int* ok) {
  if (!ok) return fail(GELATO_ERR_ARG, "null");
  CU(cudaSetDevice(device));
  DeviceBuf<double> d;
  CU(d.reserve(1));
  k_unfused_probe<<<1, 1>>>(1.0 + 0x1p-30, 1.0 - 0x1p-30, -1.0, d.get());
  double h = 1.0;
  CU(cudaMemcpy(&h, d.get(), sizeof(double), cudaMemcpyDeviceToHost));
  *ok = (h == 0.0);
  return GELATO_OK;
}

int gelato_fp64_peak(int device, double* tflops_fma, double* tflops_nofma) {
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 14;
  DeviceBuf<double> buf;
  CU(buf.reserve((size_t)blocks * threads));
  double* const d = buf.get();
  Event e0, e1;
  CU(cudaEventCreate(e0.out()));
  CU(cudaEventCreate(e1.out()));
  float ms;
  for (int pass = 0; pass < 2; pass++) {
    k_fp64_fma<<<blocks, threads>>>(d, iters);  // warm-up on pass 0
    CU(cudaDeviceSynchronize());
    CU(cudaEventRecord(e0));
    k_fp64_fma<<<blocks, threads>>>(d, iters);
    CU(cudaEventRecord(e1));
    CU(cudaEventSynchronize(e1));
    CU(cudaEventElapsedTime(&ms, e0, e1));
    if (tflops_fma) *tflops_fma = 2.0 * 8.0 * iters * (double)blocks * threads / (ms * 1e-3) / 1e12;
    k_fp64_muladd<<<blocks, threads>>>(d, iters);
    CU(cudaDeviceSynchronize());
    CU(cudaEventRecord(e0));
    k_fp64_muladd<<<blocks, threads>>>(d, iters);
    CU(cudaEventRecord(e1));
    CU(cudaEventSynchronize(e1));
    CU(cudaEventElapsedTime(&ms, e0, e1));
    if (tflops_nofma) *tflops_nofma = 2.0 * 8.0 * iters * (double)blocks * threads / (ms * 1e-3) / 1e12;
  }
  return GELATO_OK;
}

#ifdef GJ_CLOCKS
// measurement build: copy (and clear) the per-(role, warp) phase cycle sums; out[8][16][6]
int gelato_debug_clocks(unsigned long long* out) {
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpyFromSymbol(out, gj_clk_sum, sizeof(unsigned long long) * 8 * 16 * 6));
  static unsigned long long zero[8 * 16 * 6];
  CU(cudaMemcpyToSymbol(gj_clk_sum, zero, sizeof zero));
  return GELATO_OK;
}
#endif

}  // extern "C"
