// emu.cpp -- host emulator of the CUDA kernels (TEST HARNESS ONLY).
//
// Compiles gelato_b200/csrc/jobs.h (the per-thread job functions the kernels
// run) with g++ and steps through every block and thread serially: phase 1 for
// all threads of a block, then phase 2 -- the same order the block barrier
// enforces on the GPU (the Jacobian kernel has GJ_PHASES phases, the residual kernel two).  It lets the CPU-only test tier check the plan compiler
// and the kernels' index arithmetic against the oracle bit for bit, in both
// finite-difference modes, and the mesh error estimate, the path check and the path rows (mesh_error.h).  It is not
// part of the product: libgelato_b200.so has no CPU path and bench.py never
// loads this file.
#include <cstring>
#include <vector>

#include "../../gelato_b200/csrc/coord_leaves.h"
#include "../../gelato_b200/csrc/host_pool.h"
#include "../../gelato_b200/csrc/initguess.h"
#include "../../gelato_b200/csrc/output.h"
#include "../../gelato_b200/csrc/plan_host.h"

static PlanView host_view(const GelatoPlanDesc* d) {
  PlanView v;
  memset(&v, 0, sizeof v);
  planview_scalars(d, v);
  v.sec_i32 = d->sec_i32; v.sec_i64 = d->sec_i64; v.sec_f64 = d->sec_f64;
  v.d_pool = d->d_pool; v.tau_pool = d->tau_pool;
  v.wind = d->wind; v.ca = d->ca;
  v.lin_i32 = d->lin_i32; v.lin_f64 = d->lin_f64;
  v.aero_i32 = d->aero_i32; v.aero_i64 = d->aero_i64; v.aero_f64 = d->aero_f64; v.rc_aero = d->rc_aero;
  v.evt_i32 = d->evt_i32; v.evt_i64 = d->evt_i64; v.evt_f64 = d->evt_f64;
  v.packed = 0;
  return v;
}

static void attach_tables(PlanView& v, const HostTables& h) {
  v.node_rec = h.node_rec.data();
  v.jac_rec = h.jac_rec.data();
  v.aero_rows = h.aero_rows.data();
  v.n_aero_rows = (int)h.aero_rows.size();
}

static void apply_scen(PlanView& v, const GelatoScenarioDesc* sc) {
  if (!sc) return;
  if (sc->sec_f64) { v.sec_f64 = sc->sec_f64; v.sec_f64_sstride = (long long)v.S * GS_F64_COLS; }
  if (sc->wind) { v.wind = sc->wind; v.wind_sstride = (long long)v.n_wind * 3; }
  if (sc->unit_mass) v.unit_mass_scen = sc->unit_mass;
  if (sc->lin_const) v.lin_const_scen = sc->lin_const;
}

extern "C" int emu_unfused_check(void) {
  volatile double a = 1.0 + 0x1p-30, b = 1.0 - 0x1p-30, c = -1.0;
  double r = a * b + c;
  return r == 0.0;
}

extern "C" int emu_eval_residuals(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const double* x_all,
                                  double* g_all, int n_scen, const int32_t* ids) {
  if (validate_desc(d)) return -1;
  PlanView P = host_view(d);
  apply_scen(P, sc);
  HostTables h;
  build_host_tables(d, h);
  attach_tables(P, h);
  const std::vector<int32_t>& rb = h.res_blocks;
  ResScratch sm;
  for (int scen = 0; scen < n_scen; scen++) {
    const double* x = x_all + (size_t)scen * P.n_vars;
    double* g = g_all + (size_t)scen * P.n_rows;
    for (size_t b = 0; b < rb.size() / BT_COLS; b++) {
      const int32_t* bt = rb.data() + b * BT_COLS;
      memset(&sm, 0xff, sizeof sm);
      const int sid = ids ? ids[scen] : scen;
      for (int tid = 0; tid < GR_THREADS; tid++) res_block_phase0(P, sid, bt, x, tid, sm);
      for (int tid = 0; tid < GR_THREADS; tid++) res_block_phase1(P, sid, bt, x, g, tid, sm);
      for (int tid = 0; tid < GR_THREADS; tid++) res_block_phase2(P, sid, bt, x, g, tid, GR_THREADS, sm);
    }
  }
  return 0;
}

// One pass of the Jacobian blocks and vacuum nodes with finite-difference step `dx`: what launch_jacobian_pass launches.
// packed: out_all is [n_scen][n_pack] and nothing is pre-filled, else [n_scen][n_vals] from the template;  g_all != NULL:
// pair evaluation -- objfunc's rows come out of the Jacobian blocks and the linear-row blocks run too.  A sub-range (one
// problem sharded over ranks): blocks [b0, b0 + nb) and vacuum nodes [v0, v0 + nv); nb < 0: everything.
struct JacRange {
  int b0 = 0, nb = -1, v0 = 0, nv = 0;
};
static int emu_jacobian_pass(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, double dx, const double* x_all,
                             double* g_all, double* out_all, int n_scen, const int32_t* ids, int packed,
                             JacRange rg = JacRange()) {
  if (validate_desc(d)) return -1;
  PlanView P = host_view(d);
  apply_scen(P, sc);
  P.un.dx = dx;
  HostTables h;
  build_host_tables(d, h);
  attach_tables(P, h);
  PackedLayout L;
  build_packed_layout(d, L);
  P.packed = packed;
  P.n_pack = L.n_pack;
  P.sec_pk = L.sec_pk.data(); P.aero_pk = L.aero_pk.data(); P.evt_pk = L.evt_pk.data();
  const std::vector<int32_t>& jb = h.jac_blocks;
  const bool all = rg.nb < 0;
  const size_t b_lo = all ? 0 : (size_t)rg.b0;
  const size_t b_hi = b_lo + (all ? (g_all ? jb.size() / BT_COLS : (size_t)h.n_jac_main) : (size_t)rg.nb);
  const int v_lo = all ? 0 : rg.v0, v_hi = v_lo + (all ? h.n_vac : rg.nv);
  JacStore store;
  const JacScratch sm = jac_scratch(store);
  const size_t stride = packed ? (size_t)L.n_pack : (size_t)P.n_vals;
  for (int scen = 0; scen < n_scen; scen++) {
    const double* x = x_all + (size_t)scen * P.n_vars;
    double* vals = out_all + scen * stride;
    double* g = g_all ? g_all + (size_t)scen * P.n_rows : nullptr;
    const int sid = ids ? ids[scen] : scen;
    if (!packed) {
      const double* tmpl = (sc && sc->vals_template) ? sc->vals_template + (size_t)sid * P.n_vals : d->vals_template;
      memcpy(vals, tmpl, (size_t)P.n_vals * sizeof(double));
    }
    for (size_t b = b_lo; b < b_hi; b++) {
      const int32_t* bt = jb.data() + b * BT_COLS;
      /* poison the scratch so a phase that reads what no thread wrote shows up as NaN */
      memset(&store, 0xff, sizeof store);
      for (int phase = 0; phase < GJ_PHASES; phase++)
        for (int tid = 0; tid < GJ_THREADS; tid++) jac_block_phase<JR_ALL>(P, sid, bt, x, vals, g, tid, phase, sm);
    }
    /* vacuum dynamics nodes: GV_PARTS threads each (kernel k_jacobian_noair), here part after part */
    for (int k = v_lo; k < v_hi; k++) dyn_noair_node(P, sid, x, vals, g, jac_node(P, h.vac_first + k));
  }
  return 0;
}

// One Jacobian evaluation in finite-difference mode fd_mode (DESIGN.md H6): what launch_jacobian does.  Forward: one
// pass with the plan's dx.  Central: the +step pass into the caller's output (and g), the -step pass packed into
// scratch, then fd_central per x-dependent value (COO output through the packed map).  g_all == NULL: Jacobian only.
extern "C" int emu_eval_jacobian(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const double* x_all, double* g_all,
                                 double* out_all, int n_scen, const int32_t* ids, int packed, int32_t fd_mode, double step) {
  const bool central = fd_mode == GELATO_FD_CENTRAL;
  if (central && !(step > 0.0)) return -1;
  int rc = emu_jacobian_pass(d, sc, central ? step : d->dx, x_all, g_all, out_all, n_scen, ids, packed);
  if (rc || !central) return rc;
  PackedLayout L;
  build_packed_layout(d, L);
  std::vector<double> minus((size_t)n_scen * (size_t)L.n_pack);
  emu_jacobian_pass(d, sc, -step, x_all, nullptr, minus.data(), n_scen, ids, 1);
  for (int scen = 0; scen < n_scen; scen++) {
    const double* m = minus.data() + (size_t)scen * L.n_pack;
    if (packed) {
      double* out = out_all + (size_t)scen * L.n_pack;
      for (long long i = 0; i < L.n_pack; i++) out[i] = fd_central(out[i], m[i]);
    } else {
      double* out = out_all + (size_t)scen * d->n_vals;
      for (size_t i = 0; i < L.full_slot.size(); i++)
        out[L.full_slot[i]] = fd_central(out[L.full_slot[i]], L.sgn[i] * m[L.src[i]]);
    }
  }
  return 0;
}

// one problem sharded over ranks: the packed pair evaluation restricted to a block range and a vacuum-node range
// (forward differences only, as gelato_eval_pair_packed_range_dev)
extern "C" int emu_eval_pair_range(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const double* x_all, double* g_all,
                                   double* out_all, int n_scen, int b0, int nb, int v0, int nv) {
  return emu_jacobian_pass(d, sc, d->dx, x_all, g_all, out_all, n_scen, nullptr, 1, JacRange{b0, nb, v0, nv});
}
extern "C" void emu_block_counts(const GelatoPlanDesc* d, int* n_blocks_pair, int* n_vac) {
  HostTables h;
  build_host_tables(d, h);
  *n_blocks_pair = (int)(h.jac_blocks.size() / BT_COLS);
  *n_vac = h.n_vac;
}

// ---- test grids: mesh error estimate, path check and path rows (mesh_error.h; DESIGN.md section 11) ----
// What every entry point on a test grid starts from: the plan's view with the scenario blocks sc, the LGR nodes of
// each section and grid g's sections and test points (plan_host.h: build_mesh_grid, what the grid setters keep).
struct GridCall {
  PlanView P;
  std::vector<int32_t> n;
  std::vector<MeshSec> ms;
  std::vector<MeshPt> mp;
};
// NULL or why the call is refused: the description fails validate_desc, g == NULL (no grid set: `no_grid`) or the grid
// fails build_mesh_grid
static const char* grid_call(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const GelatoMeshGridDesc* g,
                             const char* no_grid, GridCall& c) {
  if (const char* why = validate_desc(d)) return why;
  if (!g) return no_grid;
  c.P = host_view(d);
  apply_scen(c.P, sc);
  c.n.resize(d->n_sections);
  for (int i = 0; i < d->n_sections; i++) c.n[i] = d->sec_i32[i * GS_I32_COLS + GS_N];
  return build_mesh_grid(g, c.n.data(), d->n_sections, c.ms, c.mp);
}

// NULL or why gelato_plan_set_mesh_grid refuses the grid
extern "C" const char* emu_check_mesh_grid(const GelatoPlanDesc* d, const GelatoMeshGridDesc* g) {
  GridCall c;
  return grid_call(d, nullptr, g, GELATO_NO_MESH_GRID, c);
}

// err_all: [n_scen][S][11]; what k_mesh_points (every test point) and then k_mesh_error (every section and state
// component) compute.  Returns NULL or why gelato_eval_mesh_error refuses the call (g == NULL: no grid set).
extern "C" const char* emu_eval_mesh_error(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const GelatoMeshGridDesc* g,
                                           const double* x_all, double* err_all, int n_scen) {
  GridCall c;
  if (const char* why = grid_call(d, sc, g, GELATO_NO_MESH_GRID, c)) return why;
  const PlanView& P = c.P;
  std::vector<double> pts(c.mp.size() * MESH_PT);
  for (int scen = 0; scen < n_scen; scen++) {
    const double* x = x_all + (size_t)scen * P.n_vars;
    for (size_t k = 0; k < c.mp.size(); k++) {
      const MeshPt q = c.mp[k];
      double* out = pts.data() + k * MESH_PT;
      mesh_point(P, scen, x, q.sec, mesh_tabs(g->pool, c.ms[q.sec], c.n[q.sec]), q.l, out, out + MESH_STATE);
    }
    for (int i = 0; i < P.S; i++)
      for (int k = 0; k < MESH_STATE; k++)
        err_all[((size_t)scen * P.S + i) * MESH_STATE + k] = mesh_component(
            P, x, i, mesh_tabs(g->pool, c.ms[i], c.n[i]), c.ms[i].m, pts.data() + (size_t)c.ms[i].pt0 * MESH_PT, k);
  }
  return nullptr;
}

// res_all / at_all: [n_scen][n_aero]; what k_path_points (every test point of the aero jobs over a whole section) and
// then k_path_min (every aero job) compute.  Returns NULL or why gelato_eval_path_check refuses the call (g == NULL: no
// grid set).
extern "C" const char* emu_eval_path_check(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const GelatoMeshGridDesc* g,
                                           const double* x_all, double* res_all, int32_t* at_all, int n_scen) {
  GridCall c;
  if (const char* why = grid_call(d, sc, g, GELATO_NO_MESH_GRID, c)) return why;
  std::vector<PathPt> pp;
  std::vector<int32_t> job0;
  if (const char* why = build_path_points(d->aero_i32, d->n_aero, c.ms, pp, job0)) return why;
  std::vector<double> r(pp.size());
  for (int scen = 0; scen < n_scen; scen++) {
    const double* x = x_all + (size_t)scen * c.P.n_vars;
    for (size_t k = 0; k < pp.size(); k++) {
      const int sec = d->aero_i32[pp[k].job * GA_I32_COLS + GA_SECTION];
      r[k] = mesh_path_point(c.P, scen, x, pp[k].job, mesh_tabs(g->pool, c.ms[sec], c.n[sec]), pp[k].l);
    }
    for (int j = 0; j < d->n_aero; j++)
      mesh_path_min(r.data() + job0[j], job0[j + 1] - job0[j], res_all + (size_t)scen * d->n_aero + j,
                    at_all + (size_t)scen * d->n_aero + j);
  }
  return nullptr;
}

// The path rows of grid g (plan_host.h: build_path_rows, what gelato_plan_set_path_rows keeps): *n_rows, *n_vals and,
// where the arrays are not NULL, each row's job, test point and offsets [n_rows][PR_OFFS] (gelato_plan_path_rows).
// Returns NULL or why gelato_plan_set_path_rows refuses the grid.
extern "C" const char* emu_plan_path_rows(const GelatoPlanDesc* d, const GelatoMeshGridDesc* g, int32_t* n_rows,
                                          int64_t* n_vals, int32_t* job, int32_t* l, int64_t* off) {
  GridCall c;
  std::vector<PathRow> rows;
  long long nv = 0;
  if (const char* why = grid_call(d, nullptr, g, GELATO_NO_PATH_ROWS, c)) return why;
  if (const char* why = build_path_rows(d->aero_i32, d->n_aero, c.n.data(), c.ms, g->pool, rows, &nv)) return why;
  *n_rows = (int32_t)rows.size();
  *n_vals = nv;
  for (size_t k = 0; k < rows.size(); k++) {
    if (job) job[k] = rows[k].job;
    if (l) l[k] = rows[k].l;
    if (off)
      for (int i = 0; i < PR_OFFS; i++) off[k * PR_OFFS + i] = rows[k].off[i];
  }
  return nullptr;
}

// g_all: [n_scen][n_rows], vals_all: [n_scen][n_vals], either may be NULL; what k_path_rows computes, lane by lane, in
// finite-difference mode `fd_mode` (gelato_plan_set_fd) with step `step` (forward: the plan's dx).  Returns NULL or why
// gelato_eval_path_rows refuses the call (g == NULL: no path rows set).
extern "C" const char* emu_eval_path_rows(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const GelatoMeshGridDesc* g,
                                          const double* x_all, double* g_all, double* vals_all, int n_scen, int32_t fd_mode,
                                          double step) {
  GridCall c;
  std::vector<PathRow> rows;
  long long nv = 0;
  if (const char* why = grid_call(d, sc, g, GELATO_NO_PATH_ROWS, c)) return why;
  if (const char* why = build_path_rows(d->aero_i32, d->n_aero, c.n.data(), c.ms, g->pool, rows, &nv)) return why;
  const PlanView& P = c.P;
  const int central = fd_mode == GELATO_FD_CENTRAL;
  const double dx = central ? step : P.un.dx;
  for (int scen = 0; scen < n_scen; scen++) {
    const double* x = x_all + (size_t)scen * P.n_vars;
    for (size_t k = 0; k < rows.size(); k++) {
      const PathRow& pr = rows[k];
      const int sec = d->aero_i32[pr.job * GA_I32_COLS + GA_SECTION];
      const MeshTabs tb = mesh_tabs(g->pool, c.ms[sec], c.n[sec]);
      double v[10];
      mesh_path_state(P, x, sec, tb, pr.l, v);
      const double f0 = path_lane_f(P, scen, x, pr.job, tb, pr.l, v, 0, 0.0);
      if (g_all) g_all[(size_t)scen * rows.size() + k] = 1.0 - f0;
      if (!vals_all) continue;
      for (int lane = 1; lane <= 12; lane++) {
        if (pr.off[PR_QUAT] < 0 && lane >= 7 && lane <= 10) continue;
        const double q = path_lane_quot(P, scen, x, pr.job, tb, pr.l, v, lane, f0, central, dx);
        path_lane_store(pr, tb.P + (long long)pr.l * (c.n[sec] + 1), c.n[sec], lane, q, vals_all + (size_t)scen * nv);
      }
    }
  }
  return nullptr;
}

// packed layout of a plan: returns n_pack; with non-NULL arrays also the map of the n_xdep COO slots
extern "C" long long emu_packed_map(const GelatoPlanDesc* d, int64_t* full_slot, int64_t* src, double* sgn) {
  if (validate_desc(d)) return -1;
  PackedLayout L;
  build_packed_layout(d, L);
  if (full_slot && src && sgn)
    for (size_t i = 0; i < L.full_slot.size(); i++) {
      full_slot[i] = L.full_slot[i];
      src[i] = L.src[i];
      sgn[i] = L.sgn[i];
    }
  return L.n_pack;
}
extern "C" long long emu_n_xdep(const GelatoPlanDesc* d) {
  PackedLayout L;
  build_packed_layout(d, L);
  return (long long)L.full_slot.size();
}

// the result-table kernel's per-thread function (output.h), one call per node
extern "C" void emu_output_rows(int n, const double* mass, const double* pos, const double* vel, const double* quat,
                                const double* t, const double* thrust_vac, const double* air_area,
                                const double* nozzle_area, const double* wind, int n_wind, const double* ca, int n_ca,
                                double lat0, double lon0, double* out) {
  Tables tb;
  tb.wind = wind; tb.n_wind = n_wind; tb.ca = ca; tb.n_ca = n_ca;
  for (int i = 0; i < n; i++)
    output_row(mass[i], v3(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]), v3(vel[3 * i], vel[3 * i + 1], vel[3 * i + 2]),
               q4(quat[4 * i], quat[4 * i + 1], quat[4 * i + 2], quat[4 * i + 3]), t[i], thrust_vac[i], air_area[i],
               nozzle_area[i], tb, lat0, lon0, out + (size_t)i * GO_COLS);
}

// update mode's host side (host_pool.h): packed x-dependent slots -> the caller's Jacobian buffers
extern "C" void emu_scatter_parallel(const int64_t* idx, long long n_idx, const double* packed, double* vals,
                                     long long n_vals, int s0, int s1, int threads) {
  gelato_host::scatter_parallel(idx, n_idx, packed, vals, n_vals, s0, s1, threads);
}

extern "C" int emu_pool_workers(void) { return gelato_host::HostPool::instance().workers(); }

// the forward-simulation kernel's per-thread function (initguess.h), one call per scenario
extern "C" void emu_rocket_simulation(int n, const double* x_init, const double* events, const int32_t* zlt, int n_ev,
                                      const double* u_table, int n_u, const double* wind, int n_wind, const double* ca,
                                      int n_ca, const int64_t* ss, double t_init, const double* t_out, int n_out, double dt,
                                      double* x_out, double* u_out) {
  for (int s = 0; s < n; s++) {
    Tables tb;
    tb.wind = wind + s * ss[2]; tb.n_wind = n_wind;
    tb.ca = ca + s * ss[3]; tb.n_ca = n_ca;
    rocket_simulation_thread(x_init + s * ss[0], events + s * ss[1], zlt, n_ev, u_table, n_u, tb, t_init, t_out, n_out, dt,
                             x_out + (size_t)s * n_out * 11, u_out ? u_out + (size_t)s * n_out * 3 : nullptr);
  }
}

// the coordinate leaf kernel's per-thread function (coord_leaves.h), one call per item
extern "C" void emu_coord_leaf(int fn, int n, const double* a, int sa, const double* b, int sb, const double* t, double* out) {
  const int so = coord_leaf_n_out(fn);
  for (int i = 0; i < n; i++) {
    double av[GC_IN] = {0.0, 0.0, 0.0, 0.0}, bv[GC_IN] = {0.0, 0.0, 0.0, 0.0}, ov[GC_OUT];
    for (int k = 0; k < sa; k++) av[k] = a[(size_t)i * sa + k];
    for (int k = 0; k < sb; k++) bv[k] = b[(size_t)i * sb + k];
    coord_leaf(fn, av, bv, t ? t[i] : 0.0, ov);
    for (int k = 0; k < so; k++) out[(size_t)i * so + k] = ov[k];
  }
}
