// emu_table.cpp -- the host emulator (emu.cpp) plus the result-table user constraints (TEST HARNESS ONLY).
//
// A plan may carry table jobs (GelatoPlanDesc: n_tab, tab_*; gelato_b200/csrc/user_table.h, DESIGN.md section 10
// "a16").  This library exports emu.cpp's entry points under the same names; the three that evaluate g or Jacobian
// values run emu.cpp's evaluation and then what k_user_table computes, lane after lane, as the CUDA library launches it
// next to the other kernels: with the residual kernel, in every Jacobian pass (central mode: the +h and -h passes
// averaged like every other packed value) and in the range of a sharded evaluation that starts at block 0.  It is not
// part of the product: libgelato_b200.so has no CPU path.
#define emu_eval_residuals emu_base_eval_residuals
#define emu_eval_jacobian emu_base_eval_jacobian
#define emu_eval_pair_range emu_base_eval_pair_range
#include "emu.cpp"
#undef emu_eval_residuals
#undef emu_eval_jacobian
#undef emu_eval_pair_range

#include "../../gelato_b200/csrc/user_table.h"

// the result-table jobs of a description, with the packed offsets of layout L
static TabView host_tab(const GelatoPlanDesc* d, const PackedLayout& L) {
  TabView t;
  t.n_tab = d->n_tab;
  t.i32 = d->tab_i32; t.f64 = d->tab_f64; t.col = d->tab_col; t.aux = d->tab_aux; t.sf = d->tab_sf;
  t.pk = L.tab_pk.data();
  return t;
}

// What k_user_table computes for batch slots [0, n_scen) with step dx and output layout `packed`: every job's lanes one
// after the other (lane 0 first: the others' quotients take its values).  out_all == NULL: the pristine lane alone
// (residual); g_all == NULL: no pristine lane (Jacobian only).
static void emu_table_pass(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, double dx, const double* x_all,
                           double* g_all, double* out_all, int n_scen, const int32_t* ids, int packed) {
  PlanView P = host_view(d);
  apply_scen(P, sc);
  P.un.dx = dx;
  PackedLayout L;
  build_packed_layout(d, L);
  P.packed = packed;
  P.n_pack = L.n_pack;
  const TabView T = host_tab(d, L);
  std::vector<double> out((size_t)GT_LANES * GO_COLS);
  for (int scen = 0; scen < n_scen; scen++) {
    const double* x = x_all + (size_t)scen * P.n_vars;
    double* vals = out_all ? out_all + (size_t)scen * (packed ? (size_t)L.n_pack : (size_t)P.n_vals) : nullptr;
    double* g = g_all ? g_all + (size_t)scen * P.n_rows : nullptr;
    const int sid = ids ? ids[scen] : scen;
    for (int job = 0; job < T.n_tab; job++) {
      auto active = [&](int lane) { return lane < GT_PRISTINE ? vals != nullptr : g != nullptr; };
      for (int lane = 0; lane < GT_LANES; lane++)
        if (active(lane)) table_lane_eval(P, T, sid, x, job, lane, &out[(size_t)lane * GO_COLS]);
      for (int r = 0; r < T.i32[job * GT_I32_COLS + GT_NROW]; r++) {
        const double v0 = vals ? table_row_value(T, job, r, &out[0]) : 0.0;
        for (int lane = 0; lane < GT_LANES; lane++)
          if (active(lane))
            table_lane_store(P, T, job, r, lane, table_row_value(T, job, r, &out[(size_t)lane * GO_COLS]), v0, vals, g);
      }
    }
  }
}

extern "C" int emu_eval_residuals(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const double* x_all,
                                  double* g_all, int n_scen, const int32_t* ids) {
  const int rc = emu_base_eval_residuals(d, sc, x_all, g_all, n_scen, ids);
  if (rc == 0) emu_table_pass(d, sc, d->dx, x_all, g_all, nullptr, n_scen, ids, 0);
  return rc;
}

// emu.cpp's evaluation, then the table jobs in finite-difference mode fd_mode: forward, one pass with the plan's dx;
// central, the +step pass into the caller's output (and g), the -step pass packed into scratch and fd_central per value
// (the table rows' packed values are `direct`: value j of a row's run is aux slot j)
extern "C" int emu_eval_jacobian(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const double* x_all, double* g_all,
                                 double* out_all, int n_scen, const int32_t* ids, int packed, int32_t fd_mode, double step) {
  const int rc = emu_base_eval_jacobian(d, sc, x_all, g_all, out_all, n_scen, ids, packed, fd_mode, step);
  if (rc || d->n_tab == 0) return rc;
  const bool central = fd_mode == GELATO_FD_CENTRAL;
  emu_table_pass(d, sc, central ? step : d->dx, x_all, g_all, out_all, n_scen, ids, packed);
  if (!central) return 0;
  PackedLayout L;
  build_packed_layout(d, L);
  std::vector<double> minus((size_t)n_scen * (size_t)L.n_pack);
  emu_table_pass(d, sc, -step, x_all, nullptr, minus.data(), n_scen, ids, 1);
  for (int scen = 0; scen < n_scen; scen++) {
    const double* m = minus.data() + (size_t)scen * L.n_pack;
    double* out = out_all + (size_t)scen * (packed ? (size_t)L.n_pack : (size_t)d->n_vals);
    for (int r = 0; r < d->n_tab_rows; r++)
      for (int j = 0; j < GT_AUX; j++) {
        const long long k = (packed ? L.tab_pk[r] : d->tab_aux[r]) + j;
        out[k] = fd_central(out[k], m[L.tab_pk[r] + j]);
      }
  }
  return 0;
}

// the sharded pair evaluation: the range that starts at block 0 evaluates the table jobs
extern "C" int emu_eval_pair_range(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const double* x_all, double* g_all,
                                   double* out_all, int n_scen, int b0, int nb, int v0, int nv) {
  const int rc = emu_base_eval_pair_range(d, sc, x_all, g_all, out_all, n_scen, b0, nb, v0, nv);
  if (rc == 0 && b0 == 0 && nb > 0) emu_table_pass(d, sc, d->dx, x_all, g_all, out_all, n_scen, nullptr, 1);
  return rc;
}
