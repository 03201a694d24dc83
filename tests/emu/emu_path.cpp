// emu_path.cpp -- the host emulator (emu.cpp) plus the path check of mesh_error.h (TEST HARNESS ONLY).
//
// One library: every entry point of emu.cpp, and emu_eval_path_check, which runs what k_path_points and k_path_min
// run, through the same plan_host.h lists the library builds when a grid is set.  Loaded by tests/emu_path.py.
#include "emu.cpp"

// res_all / at_all: [n_scen][n_aero]; what k_path_points (every test point of the aero jobs over a whole section) and
// then k_path_min (every aero job) compute.  Returns NULL or why gelato_eval_path_check refuses the call (g == NULL: no
// grid set).
extern "C" const char* emu_eval_path_check(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const GelatoMeshGridDesc* g,
                                           const double* x_all, double* res_all, int32_t* at_all, int n_scen) {
  if (const char* why = validate_desc(d)) return why;
  if (!g) return GELATO_NO_MESH_GRID;
  PlanView P = host_view(d);
  apply_scen(P, sc);
  const std::vector<int32_t> n = sec_nodes(d);
  std::vector<MeshSec> ms;
  std::vector<MeshPt> mp;
  std::vector<PathPt> pp;
  std::vector<int32_t> job0;
  if (const char* why = build_mesh_grid(g, n.data(), P.S, ms, mp)) return why;
  if (const char* why = build_path_points(d->aero_i32, d->n_aero, ms, pp, job0)) return why;
  std::vector<double> r(pp.size());
  for (int scen = 0; scen < n_scen; scen++) {
    const double* x = x_all + (size_t)scen * P.n_vars;
    for (size_t k = 0; k < pp.size(); k++) {
      const int sec = d->aero_i32[pp[k].job * GA_I32_COLS + GA_SECTION];
      r[k] = mesh_path_point(P, scen, x, pp[k].job, mesh_tabs(g->pool, ms[sec], n[sec]), pp[k].l);
    }
    for (int j = 0; j < d->n_aero; j++)
      mesh_path_min(r.data() + job0[j], job0[j + 1] - job0[j], res_all + (size_t)scen * d->n_aero + j,
                    at_all + (size_t)scen * d->n_aero + j);
  }
  return nullptr;
}
