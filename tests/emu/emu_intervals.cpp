// emu_intervals.cpp -- the host emulator (emu.cpp) plus the per-interval mesh error estimate (TEST HARNESS ONLY).
//
// A mesh grid may come with interval tables (GelatoMeshGridDesc: n_int, int_m, int_base; DESIGN.md section 11,
// "h-refinement").  emu.cpp estimates each section as one interval; this file steps through what k_mesh_points and then
// k_mesh_error compute on such a grid, interval by interval, with the interval lists build_mesh_grid keeps.  It is not
// part of the product: libgelato_b200.so has no CPU path.
#include "emu.cpp"

// err_all: [n_scen][S][11], err_int: [n_scen][n_int][11], either may be NULL.  Returns NULL or why
// gelato_eval_mesh_error / gelato_eval_mesh_error_intervals refuses the call (g == NULL: no grid set).
extern "C" const char* emu_eval_mesh_error_intervals(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc,
                                                     const GelatoMeshGridDesc* g, const double* x_all, double* err_all,
                                                     double* err_int, int n_scen) {
  GridCall c;
  if (const char* why = grid_call(d, sc, g, GELATO_NO_MESH_GRID, c)) return why;
  std::vector<MeshInt> ints;
  std::vector<int32_t> int0;
  if (const char* why = build_mesh_grid(g, c.n.data(), d->n_sections, c.ms, c.mp, ints, int0)) return why;
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
      for (int k = 0; k < MESH_STATE; k++) {
        double e = 0.0;
        for (int j = int0[i]; j < int0[i + 1]; j++) {
          const double ej = mesh_component(P, x, i, mesh_tabs(g->pool, c.ms[i], c.n[i]), c.ms[i].m,
                                           pts.data() + (size_t)c.ms[i].pt0 * MESH_PT, k, ints[j]);
          if (err_int) err_int[((size_t)scen * ints.size() + j) * MESH_STATE + k] = ej;
          e = j == int0[i] ? ej : mesh_max(e, ej);
        }
        if (err_all) err_all[((size_t)scen * P.S + i) * MESH_STATE + k] = e;
      }
  }
  return nullptr;
}
