// leaf_api.cu -- batch versions of the reference's pybind11 leaf functions
// (/root/reference/src/pybind_dynamics.cpp:108-114, pybind_utils.cpp:28-48, pybind_coordinate.cpp:28-78,
// pybind_IIP.cpp:53-57, pybind_USStandardAtmosphere.cpp:28-35): one kernel launch evaluates a leaf for n
// nodes, one thread per node, with the device functions the fused kernels use (physics.h).  They serve the
// callers AROUND the NLP loop that evaluate leaves over whole trajectories (initial guess, result tables)
// and let tests compare every leaf with the oracle on its own.  Host buffers in, host buffers out.
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "../../include/gelato_b200.h"
#include "coord_leaves.h"
#include "initguess.h"
#include "output.h"

extern "C" void gelato_set_error_(const char* msg);  // gelato_b200.cu

namespace {

struct DevBuf {
  std::vector<void*> ptrs;
  ~DevBuf() { for (void* p : ptrs) cudaFree(p); }
  template <typename T>
  T* in(const T* host, size_t count, cudaError_t& err) {
    T* d = nullptr;
    if (err != cudaSuccess || count == 0) return d;
    err = cudaMalloc(&d, count * sizeof(T));
    if (err != cudaSuccess) return nullptr;
    ptrs.push_back(d);
    err = cudaMemcpy(d, host, count * sizeof(T), cudaMemcpyHostToDevice);
    return d;
  }
  double* out(size_t count, cudaError_t& err) {
    double* d = nullptr;
    if (err != cudaSuccess || count == 0) return d;
    err = cudaMalloc(&d, count * sizeof(double));
    if (err == cudaSuccess) ptrs.push_back(d);
    return d;
  }
};

int finish(cudaError_t err, double* host_out, const double* dev_out, size_t count) {
  if (err == cudaSuccess) err = cudaGetLastError();
  if (err == cudaSuccess) err = cudaMemcpy(host_out, dev_out, count * sizeof(double), cudaMemcpyDeviceToHost);
  if (err != cudaSuccess) {
    gelato_set_error_(cudaGetErrorString(err));
    return GELATO_ERR_CUDA;
  }
  return GELATO_OK;
}

inline int blocks_for(int n) { return (n + 127) / 128; }

__global__ void k_leaf_dynamics_velocity(int n, const double* mass_e, const double* pos_e, const double* vel_e,
                                         const double* quat, const double* t, SecParam sp, Units un, Tables tb,
                                         double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Vec3 f = rhs_velocity_air(mass_e[i], v3(pos_e[3 * i], pos_e[3 * i + 1], pos_e[3 * i + 2]),
                            v3(vel_e[3 * i], vel_e[3 * i + 1], vel_e[3 * i + 2]),
                            q4(quat[4 * i], quat[4 * i + 1], quat[4 * i + 2], quat[4 * i + 3]), t[i], sp, un, tb);
  out[3 * i] = f.x; out[3 * i + 1] = f.y; out[3 * i + 2] = f.z;
}

__global__ void k_leaf_dynamics_velocity_noair(int n, const double* mass_e, const double* pos_e, const double* quat,
                                               SecParam sp, Units un, double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Vec3 f = rhs_velocity_noair(mass_e[i], v3(pos_e[3 * i], pos_e[3 * i + 1], pos_e[3 * i + 2]),
                              q4(quat[4 * i], quat[4 * i + 1], quat[4 * i + 2], quat[4 * i + 3]), sp, un);
  out[3 * i] = f.x; out[3 * i + 1] = f.y; out[3 * i + 2] = f.z;
}

__global__ void k_leaf_dynamics_quaternion(int n, const double* quat, const double* u_e, double unit_u, double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Quat d = rhs_quaternion(q4(quat[4 * i], quat[4 * i + 1], quat[4 * i + 2], quat[4 * i + 3]), u_e[2 * i],
                          u_e[2 * i + 1], unit_u);
  out[4 * i] = d.w; out[4 * i + 1] = d.x; out[4 * i + 2] = d.y; out[4 * i + 3] = d.z;
}

__global__ void k_leaf_aero(int kind, int n, const double* pos, const double* vel, const double* quat,
                            const double* t, Tables tb, double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (kind == 4) { /* wind_ned(altitude, table): t[] carries the altitudes (wrapper_utils.hpp:82-87) */
    out[3 * i] = interp_table(t[i], tb.wind, tb.wind + 1, tb.n_wind, 3);
    out[3 * i + 1] = interp_table(t[i], tb.wind, tb.wind + 2, tb.n_wind, 3);
    out[3 * i + 2] = 0.0;
    return;
  }
  Quat q = q4(1.0, 0.0, 0.0, 0.0);
  if (quat) q = q4(quat[4 * i], quat[4 * i + 1], quat[4 * i + 2], quat[4 * i + 3]);
  const Vec3 p = v3(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]), v = v3(vel[3 * i], vel[3 * i + 1], vel[3 * i + 2]);
  if (kind == 3) { /* angle_of_attack_ab_rad -> (pitch-plane, yaw-plane) (wrapper_utils.hpp:125-148) */
    angle_of_attack_ab(p, v, q, t[i], tb, out + 2 * i);
    return;
  }
  out[i] = aero_quantity(kind, p, v, q, t[i], tb);
}

__global__ void k_leaf_eci2geodetic(int n, const double* pos, const double* t, double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Vec3 g = eci2geodetic_deg(v3(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]), t[i]);
  out[3 * i] = g.x; out[3 * i + 1] = g.y; out[3 * i + 2] = g.z;
}

__global__ void k_leaf_iip(int n, const double* pos_ecef, const double* vel_ecef, int fill_na, double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Vec3 g = iip_faa_deg(v3(pos_ecef[3 * i], pos_ecef[3 * i + 1], pos_ecef[3 * i + 2]),
                       v3(vel_ecef[3 * i], vel_ecef[3 * i + 1], vel_ecef[3 * i + 2]));
  /* pybind_IIP.cpp:38-45: with fill_na = false an all-zero "no solution" becomes NaN */
  if (!fill_na && g.x == 0.0 && g.y == 0.0 && g.z == 0.0) g.x = g.y = g.z = gm_nan();
  out[3 * i] = g.x; out[3 * i + 1] = g.y; out[3 * i + 2] = g.z;
}

__global__ void k_leaf_gravity(int n, const double* pos, double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Vec3 g = gravity_eci(v3(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]));
  out[3 * i] = g.x; out[3 * i + 1] = g.y; out[3 * i + 2] = g.z;
}

/* out[i][5] = geopotential_altitude(z), airtemperature_at(z), airpressure_at(z), airdensity_at(z),
 * speed_of_sound(z), each applied to z as given (pybind_USStandardAtmosphere.cpp:28-35) */
__global__ void k_leaf_atmosphere(int n, const double* z, double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  AirState s = us76(z[i], 3);
  out[5 * i] = geopotential_altitude(z[i]);
  out[5 * i + 1] = s.T;
  out[5 * i + 2] = s.P;
  out[5 * i + 3] = s.rho;
  out[5 * i + 4] = s.a;
}

/* one row of the reference's result table per thread (output.h) */
__global__ void k_leaf_output_table(int n, const double* mass, const double* pos, const double* vel, const double* quat,
                                    const double* t, const double* thrust_vac, const double* air_area,
                                    const double* nozzle_area, Tables tb, double lat0, double lon0, double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double row[GO_COLS];
  output_row(mass[i], v3(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]), v3(vel[3 * i], vel[3 * i + 1], vel[3 * i + 2]),
             q4(quat[4 * i], quat[4 * i + 1], quat[4 * i + 2], quat[4 * i + 3]), t[i], thrust_vac[i], air_area[i],
             nozzle_area[i], tb, lat0, lon0, row);
  for (int k = 0; k < GO_COLS; k++) out[(size_t)i * GO_COLS + k] = row[k];
}


// forward-simulation initial guess (initguess.h): one thread per scenario walks the whole event schedule.  The
// scenarios of a dispersed batch differ in their initial state, event rows and tables; the mesh times, the rate
// table and the zero-lift-turn flags are shared.
struct InitStrides {
  long long x_init, events, wind, ca;  // doubles between consecutive scenarios; 0 = one copy shared by all
};
__global__ void k_init_rocket_simulation(int n_scen, const double* x_init, const double* ev, const int32_t* zlt, int n_ev,
                                         const double* u_table, int n_u, const double* wind, int n_wind, const double* ca,
                                         int n_ca, InitStrides ss, double t_init, const double* t_out, int n_out, double dt,
                                         double* x_out, double* u_out) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_scen) return;
  Tables tb;
  tb.wind = wind + s * ss.wind; tb.n_wind = n_wind;
  tb.ca = ca + s * ss.ca; tb.n_ca = n_ca;
  rocket_simulation_thread(x_init + s * ss.x_init, ev + s * ss.events, zlt, n_ev, u_table, n_u, tb, t_init, t_out, n_out, dt,
                           x_out + (size_t)s * n_out * 11, u_out ? u_out + (size_t)s * n_out * 3 : nullptr);
}


// the coordinate_c / utils_c leaves that are not on the NLP path (coord_leaves.h), one thread per item
__global__ void k_leaf_coordinate(int fn, int n, const double* a, int sa, const double* b, int sb, const double* t, double* out,
                                  int so) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double av[GC_IN] = {0.0, 0.0, 0.0, 0.0}, bv[GC_IN] = {0.0, 0.0, 0.0, 0.0}, ov[GC_OUT];
  for (int k = 0; k < sa; k++) av[k] = a[(size_t)i * sa + k];
  for (int k = 0; k < sb; k++) bv[k] = b[(size_t)i * sb + k];
  coord_leaf(fn, av, bv, t ? t[i] : 0.0, ov);
  for (int k = 0; k < so; k++) out[(size_t)i * so + k] = ov[k];
}


}  // namespace

extern "C" {

#define LEAF_PROLOGUE                                                          \
  if (n <= 0) { gelato_set_error_("n must be positive"); return GELATO_ERR_ARG; } \
  cudaError_t err = cudaSetDevice(device);                                     \
  DevBuf buf;

// interp_interval / np_interp (physics.h) read rows k and k + 1 of a table: one row is refused, as
// gelato_plan_create refuses it (plan_host.h: validate_desc)
#define LEAF_TABLE_ROWS(name, table, rows)                                              \
  if (!(table) || (rows) < 2) {                                                        \
    gelato_set_error_(name ": " #table " table needs at least two rows");               \
    return GELATO_ERR_ARG;                                                             \
  }

int gelato_leaf_dynamics_velocity(int device, int32_t n, const double* mass_e, const double* pos_e,
                                  const double* vel_e, const double* quat, const double* t, const double* param5,
                                  const double* wind, int32_t n_wind, const double* ca, int32_t n_ca,
                                  const double* units3, double* out) {
  LEAF_PROLOGUE
  LEAF_TABLE_ROWS("gelato_leaf_dynamics_velocity", wind, n_wind)
  LEAF_TABLE_ROWS("gelato_leaf_dynamics_velocity", ca, n_ca)
  SecParam sp{param5[0], param5[1], param5[2], param5[4]};
  Units un{units3[0], units3[1], units3[2], 1.0, 1.0, 0.0};
  Tables tb;
  tb.wind = buf.in(wind, (size_t)n_wind * 3, err); tb.n_wind = n_wind;
  tb.ca = buf.in(ca, (size_t)n_ca * 2, err); tb.n_ca = n_ca;
  const double* dm = buf.in(mass_e, n, err);
  const double* dp = buf.in(pos_e, (size_t)3 * n, err);
  const double* dv = buf.in(vel_e, (size_t)3 * n, err);
  const double* dq = buf.in(quat, (size_t)4 * n, err);
  const double* dt = buf.in(t, n, err);
  double* d_out = buf.out((size_t)3 * n, err);
  if (err == cudaSuccess) k_leaf_dynamics_velocity<<<blocks_for(n), 128>>>(n, dm, dp, dv, dq, dt, sp, un, tb, d_out);
  return finish(err, out, d_out, (size_t)3 * n);
}

int gelato_leaf_dynamics_velocity_noair(int device, int32_t n, const double* mass_e, const double* pos_e,
                                        const double* quat, const double* param5, const double* units3, double* out) {
  LEAF_PROLOGUE
  SecParam sp{param5[0], param5[1], param5[2], param5[4]};
  Units un{units3[0], units3[1], units3[2], 1.0, 1.0, 0.0};
  const double* dm = buf.in(mass_e, n, err);
  const double* dp = buf.in(pos_e, (size_t)3 * n, err);
  const double* dq = buf.in(quat, (size_t)4 * n, err);
  double* d_out = buf.out((size_t)3 * n, err);
  if (err == cudaSuccess) k_leaf_dynamics_velocity_noair<<<blocks_for(n), 128>>>(n, dm, dp, dq, sp, un, d_out);
  return finish(err, out, d_out, (size_t)3 * n);
}

int gelato_leaf_dynamics_quaternion(int device, int32_t n, const double* quat, const double* u_e, double unit_u,
                                    double* out) {
  LEAF_PROLOGUE
  const double* dq = buf.in(quat, (size_t)4 * n, err);
  const double* du = buf.in(u_e, (size_t)2 * n, err);
  double* d_out = buf.out((size_t)4 * n, err);
  if (err == cudaSuccess) k_leaf_dynamics_quaternion<<<blocks_for(n), 128>>>(n, dq, du, unit_u, d_out);
  return finish(err, out, d_out, (size_t)4 * n);
}

int gelato_leaf_aero(int device, int32_t kind, int32_t n, const double* pos, const double* vel, const double* quat,
                     const double* t, const double* wind, int32_t n_wind, double* out) {
  LEAF_PROLOGUE
  const bool state = kind != 4;  // kind 4 (wind_ned) reads the altitudes in t and the table only
  LEAF_TABLE_ROWS("gelato_leaf_aero", wind, n_wind)
  if (kind < 0 || kind > 4 || !t || !out || (state && (!pos || !vel)) ||
      ((kind == 0 || kind == 2 || kind == 3) && !quat)) {
    gelato_set_error_("gelato_leaf_aero: bad kind, missing quaternion or null buffer");
    return GELATO_ERR_ARG;
  }
  Tables tb;
  tb.wind = buf.in(wind, (size_t)n_wind * 3, err); tb.n_wind = n_wind;
  tb.ca = nullptr; tb.n_ca = 0;
  const double* dp = state ? buf.in(pos, (size_t)3 * n, err) : nullptr;
  const double* dv = state ? buf.in(vel, (size_t)3 * n, err) : nullptr;
  const double* dq = (state && quat) ? buf.in(quat, (size_t)4 * n, err) : nullptr;
  const double* dt = buf.in(t, n, err);
  const size_t width = kind == 3 ? 2 : kind == 4 ? 3 : 1;
  double* d_out = buf.out(width * n, err);
  if (err == cudaSuccess) k_leaf_aero<<<blocks_for(n), 128>>>(kind, n, dp, dv, dq, dt, tb, d_out);
  return finish(err, out, d_out, width * n);
}

int gelato_leaf_eci2geodetic(int device, int32_t n, const double* pos_eci, const double* t, double* out) {
  LEAF_PROLOGUE
  const double* dp = buf.in(pos_eci, (size_t)3 * n, err);
  const double* dt = buf.in(t, n, err);
  double* d_out = buf.out((size_t)3 * n, err);
  if (err == cudaSuccess) k_leaf_eci2geodetic<<<blocks_for(n), 128>>>(n, dp, dt, d_out);
  return finish(err, out, d_out, (size_t)3 * n);
}

int gelato_leaf_iip(int device, int32_t n, const double* pos_ecef, const double* vel_ecef, int32_t fill_na,
                    double* out) {
  LEAF_PROLOGUE
  const double* dp = buf.in(pos_ecef, (size_t)3 * n, err);
  const double* dv = buf.in(vel_ecef, (size_t)3 * n, err);
  double* d_out = buf.out((size_t)3 * n, err);
  if (err == cudaSuccess) k_leaf_iip<<<blocks_for(n), 128>>>(n, dp, dv, fill_na, d_out);
  return finish(err, out, d_out, (size_t)3 * n);
}

int gelato_leaf_gravity(int device, int32_t n, const double* pos_eci, double* out) {
  LEAF_PROLOGUE
  const double* dp = buf.in(pos_eci, (size_t)3 * n, err);
  double* d_out = buf.out((size_t)3 * n, err);
  if (err == cudaSuccess) k_leaf_gravity<<<blocks_for(n), 128>>>(n, dp, d_out);
  return finish(err, out, d_out, (size_t)3 * n);
}

int gelato_leaf_output_table(int device, int32_t n, const double* mass, const double* pos, const double* vel,
                             const double* quat, const double* t, const double* thrust_vac, const double* air_area,
                             const double* nozzle_area, const double* wind, int32_t n_wind, const double* ca, int32_t n_ca,
                             double launch_lat_deg, double launch_lon_deg, double* out) {
  LEAF_PROLOGUE
  LEAF_TABLE_ROWS("gelato_leaf_output_table", wind, n_wind)
  LEAF_TABLE_ROWS("gelato_leaf_output_table", ca, n_ca)
  Tables tb;
  tb.wind = buf.in(wind, (size_t)n_wind * 3, err); tb.n_wind = n_wind;
  tb.ca = buf.in(ca, (size_t)n_ca * 2, err); tb.n_ca = n_ca;
  const double* dm = buf.in(mass, n, err);
  const double* dp = buf.in(pos, (size_t)3 * n, err);
  const double* dv = buf.in(vel, (size_t)3 * n, err);
  const double* dq = buf.in(quat, (size_t)4 * n, err);
  const double* dt = buf.in(t, n, err);
  const double* d1 = buf.in(thrust_vac, n, err);
  const double* d2 = buf.in(air_area, n, err);
  const double* d3 = buf.in(nozzle_area, n, err);
  double* d_out = buf.out((size_t)GO_COLS * n, err);
  if (err == cudaSuccess)
    k_leaf_output_table<<<blocks_for(n), 128>>>(n, dm, dp, dv, dq, dt, d1, d2, d3, tb, launch_lat_deg, launch_lon_deg, d_out);
  return finish(err, out, d_out, (size_t)GO_COLS * n);
}

int gelato_leaf_atmosphere(int device, int32_t n, const double* altitude, double* out) {
  LEAF_PROLOGUE
  const double* dz = buf.in(altitude, n, err);
  double* d_out = buf.out((size_t)5 * n, err);
  if (err == cudaSuccess) k_leaf_atmosphere<<<blocks_for(n), 128>>>(n, dz, d_out);
  return finish(err, out, d_out, (size_t)5 * n);
}

int gelato_init_rocket_simulation(int device, int32_t n, const double* x_init, const double* events, const int32_t* zlt,
                                  int32_t n_ev, const double* u_table, int32_t n_u, const double* wind, int32_t n_wind,
                                  const double* ca, int32_t n_ca, const int64_t* scenario_strides, double t_init,
                                  const double* t_out, int32_t n_out, double dt, double* x_out, double* u_out) {
  LEAF_PROLOGUE
  if (!x_init || !events || !zlt || !u_table || !wind || !ca || !t_out || !x_out) {
    gelato_set_error_("rocket_simulation: null buffer");
    return GELATO_ERR_ARG;
  }
  LEAF_TABLE_ROWS("rocket_simulation", wind, n_wind)
  LEAF_TABLE_ROWS("rocket_simulation", ca, n_ca)
  if (n_ev <= 0 || n_u <= 0 || n_out <= 0 || !(dt > 0.0) || !scenario_strides) {
    gelato_set_error_("rocket_simulation: empty table, no output time or non-positive dt");
    return GELATO_ERR_ARG;
  }
  const InitStrides ss = {scenario_strides[0], scenario_strides[1], scenario_strides[2], scenario_strides[3]};
  const long long need[4] = {11, (long long)n_ev * GI_COLS, (long long)n_wind * 3, (long long)n_ca * 2};
  const long long have[4] = {ss.x_init, ss.events, ss.wind, ss.ca};
  size_t count[4];
  for (int k = 0; k < 4; k++) {
    if (have[k] != 0 && have[k] < need[k]) {
      gelato_set_error_("rocket_simulation: a scenario stride is shorter than one scenario's table");
      return GELATO_ERR_ARG;
    }
    count[k] = have[k] ? (size_t)have[k] * (n - 1) + need[k] : (size_t)need[k];
  }
  for (int i = 1; i < n_out; i++)
    if (!(t_out[i] >= t_out[i - 1])) {
      gelato_set_error_("rocket_simulation: output times must ascend");
      return GELATO_ERR_ARG;
    }
  const double* dx = buf.in(x_init, count[0], err);
  const double* de = buf.in(events, count[1], err);
  const double* dw = buf.in(wind, count[2], err);
  const double* dc = buf.in(ca, count[3], err);
  const int32_t* dz = buf.in(zlt, (size_t)n_ev, err);
  const double* du = buf.in(u_table, (size_t)n_u * 4, err);
  const double* dto = buf.in(t_out, (size_t)n_out, err);
  double* d_out = buf.out((size_t)n * n_out * 11, err);
  double* d_uout = u_out ? buf.out((size_t)n * n_out * 3, err) : nullptr;
  // 32 threads per block: a batch of a few thousand scenarios then covers every SM (each thread is one long serial
  // integration, so the launch is latency-bound and wants as many SMs as it can touch)
  if (err == cudaSuccess)
    k_init_rocket_simulation<<<(n + 31) / 32, 32>>>(n, dx, de, dz, n_ev, du, n_u, dw, n_wind, dc, n_ca, ss, t_init, dto, n_out,
                                                    dt, d_out, d_uout);
  if (err == cudaSuccess) err = cudaDeviceSynchronize();
  if (err == cudaSuccess && u_out) err = cudaMemcpy(u_out, d_uout, (size_t)n * n_out * 3 * sizeof(double), cudaMemcpyDeviceToHost);
  return finish(err, x_out, d_out, (size_t)n * n_out * 11);
}

int gelato_leaf_coordinate(int device, int32_t fn, int32_t n, const double* a, int32_t a_width, const double* b, int32_t b_width,
                           const double* t, double* out) {
  LEAF_PROLOGUE
  if (fn < 0 || fn >= GC_N_FUNCTIONS || a_width < 0 || a_width > GC_IN || b_width < 0 || b_width > GC_IN || !out ||
      (a_width > 0 && !a) || (b_width > 0 && !b)) {
    gelato_set_error_("gelato_leaf_coordinate: unknown function code, width outside 0..9 or null buffer");
    return GELATO_ERR_ARG;
  }
  const int so = coord_leaf_n_out(fn);
  const double* da = buf.in(a, (size_t)n * a_width, err);
  const double* db = buf.in(b, (size_t)n * b_width, err);
  const double* dt = t ? buf.in(t, (size_t)n, err) : nullptr;
  double* d_out = buf.out((size_t)n * so, err);
  if (err == cudaSuccess) k_leaf_coordinate<<<blocks_for(n), 128>>>(fn, n, da, a_width, db, b_width, dt, d_out, so);
  return finish(err, out, d_out, (size_t)n * so);
}

}  // extern "C"
