// emu_mesh.cpp -- host emulator of the mesh error estimate (TEST HARNESS ONLY; DESIGN.md section 11).
//
// What gelato_b200.cu: k_mesh_points and k_mesh_error compute, stepped on the host with the kernels' per-thread code
// (mesh_error.h): every test point of every section, then every (section, state component).  It builds on the
// emulator of emu.cpp (plan view, scenario blocks), compiled into this library.
#include "emu.cpp"
#include "../../gelato_b200/csrc/mesh_error.h"

// err_all: [n_scen][S][11]; the grid is taken as given (gelato_plan_set_mesh_grid checks it on the device path).
extern "C" int emu_mesh_error(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const GelatoMeshGridDesc* g,
                              const double* x_all, double* err_all, int n_scen) {
  if (validate_desc(d)) return -1;
  PlanView P = host_view(d);
  apply_scen(P, sc);
  const int S = P.S;
  std::vector<MeshSec> ms(S);
  int n_pts = 0;
  for (int i = 0; i < S; i++) {
    ms[i].m = g->m[i];
    ms[i].pt0 = n_pts;
    ms[i].off = g->off[i];
    n_pts += g->m[i];
  }
  std::vector<double> pts((size_t)n_pts * MESH_PT);
  for (int scen = 0; scen < n_scen; scen++) {
    const double* x = x_all + (size_t)scen * P.n_vars;
    for (int i = 0; i < S; i++) {
      const MeshTabs tb = mesh_tabs(g->pool, ms[i], d->sec_i32[i * GS_I32_COLS + GS_N]);
      for (int l = 0; l < ms[i].m; l++) {
        double* q = pts.data() + (size_t)(ms[i].pt0 + l) * MESH_PT;
        mesh_point(P, scen, x, i, tb, l, q, q + MESH_STATE);
      }
    }
    for (int i = 0; i < S; i++) {
      const MeshTabs tb = mesh_tabs(g->pool, ms[i], d->sec_i32[i * GS_I32_COLS + GS_N]);
      for (int c = 0; c < MESH_STATE; c++)
        err_all[((size_t)scen * S + i) * MESH_STATE + c] =
            mesh_component(P, x, i, tb, ms[i].m, pts.data() + (size_t)ms[i].pt0 * MESH_PT, c);
    }
  }
  return 0;
}
