// emu_path_rows.cpp -- the host emulator with the path check (emu_path.cpp) plus the path rows (TEST HARNESS ONLY).
//
// One library: every entry point of emu_path.cpp, and emu_path_rows / emu_eval_path_rows, which run what
// gelato_plan_set_path_rows keeps (plan_host.h: build_path_rows) and what k_path_rows computes, lane by lane, through the
// per-thread functions of mesh_error.h.  Loaded by tests/emu_path_rows.py.
#include "emu_path.cpp"

// The path rows of grid g (plan_host.h: build_path_rows, what gelato_plan_set_path_rows keeps): *n_rows, *n_vals and,
// where the arrays are not NULL, each row's job, test point and offsets [n_rows][PR_OFFS] (gelato_plan_path_rows).
// Returns NULL or why gelato_plan_set_path_rows refuses the grid.
extern "C" const char* emu_path_rows(const GelatoPlanDesc* d, const GelatoMeshGridDesc* g, int32_t* n_rows, int64_t* n_vals,
                                     int32_t* job, int32_t* l, int64_t* off) {
  if (const char* why = validate_desc(d)) return why;
  const std::vector<int32_t> n = sec_nodes(d);
  std::vector<MeshSec> ms;
  std::vector<MeshPt> mp;
  std::vector<PathRow> rows;
  long long nv = 0;
  if (const char* why = build_mesh_grid(g, n.data(), d->n_sections, ms, mp)) return why;
  if (const char* why = build_path_rows(d->aero_i32, d->n_aero, n.data(), ms, g->pool, rows, &nv)) return why;
  *n_rows = (int32_t)rows.size();
  *n_vals = nv;
  for (size_t k = 0; k < rows.size(); k++) {
    if (job) job[k] = rows[k].job;
    if (l) l[k] = rows[k].l;
    if (off)
      for (int c = 0; c < PR_OFFS; c++) off[k * PR_OFFS + c] = rows[k].off[c];
  }
  return nullptr;
}

// g_all: [n_scen][n_rows], vals_all: [n_scen][n_vals], either may be NULL; what k_path_rows computes, lane by lane, in
// finite-difference mode `fd_mode` (gelato_plan_set_fd) with step `step` (forward: the plan's dx).  Returns NULL or why
// gelato_eval_path_rows refuses the call (g == NULL: no path rows set).
extern "C" const char* emu_eval_path_rows(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const GelatoMeshGridDesc* g,
                                          const double* x_all, double* g_all, double* vals_all, int n_scen, int32_t fd_mode,
                                          double step) {
  if (const char* why = validate_desc(d)) return why;
  if (!g) return GELATO_NO_PATH_ROWS;
  PlanView P = host_view(d);
  apply_scen(P, sc);
  const std::vector<int32_t> n = sec_nodes(d);
  std::vector<MeshSec> ms;
  std::vector<MeshPt> mp;
  std::vector<PathRow> rows;
  long long nv = 0;
  if (const char* why = build_mesh_grid(g, n.data(), P.S, ms, mp)) return why;
  if (const char* why = build_path_rows(d->aero_i32, d->n_aero, n.data(), ms, g->pool, rows, &nv)) return why;
  const int central = fd_mode == GELATO_FD_CENTRAL;
  const double dx = central ? step : P.un.dx;
  for (int scen = 0; scen < n_scen; scen++) {
    const double* x = x_all + (size_t)scen * P.n_vars;
    for (size_t k = 0; k < rows.size(); k++) {
      const PathRow& pr = rows[k];
      const int sec = d->aero_i32[pr.job * GA_I32_COLS + GA_SECTION];
      const MeshTabs tb = mesh_tabs(g->pool, ms[sec], n[sec]);
      double v[10];
      mesh_path_state(P, x, sec, tb, pr.l, v);
      const double f0 = path_lane_f(P, scen, x, pr.job, tb, pr.l, v, 0, 0.0);
      if (g_all) g_all[(size_t)scen * rows.size() + k] = 1.0 - f0;
      if (!vals_all) continue;
      for (int lane = 1; lane <= 12; lane++) {
        if (pr.off[PR_QUAT] < 0 && lane >= 7 && lane <= 10) continue;
        const double q = path_lane_quot(P, scen, x, pr.job, tb, pr.l, v, lane, f0, central, dx);
        path_lane_store(pr, tb.P + (long long)pr.l * (n[sec] + 1), n[sec], lane, q, vals_all + (size_t)scen * nv);
      }
    }
  }
  return nullptr;
}
