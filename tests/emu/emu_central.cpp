// emu_central.cpp -- host emulator of the central-difference Jacobian (TEST HARNESS ONLY; DESIGN.md H6).
//
// What gelato_b200.cu: launch_jacobian does in GELATO_FD_CENTRAL mode, stepped on the host with the kernels'
// per-thread code: the forward protocol with step +h into the caller's output (and g of a pair evaluation), the
// same with -h packed into scratch, then jobs.h: fd_central per x-dependent value (COO output through the packed map).
// It builds on the emulator of emu.cpp (plan set-up, block order), compiled into this library.
#include "emu.cpp"

// One pass of the Jacobian blocks and vacuum nodes with finite-difference step `dx` (the plan's dx is not used, so
// the -h pass needs no plan description with a negative dx, which validate_desc refuses).
static void central_pass(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const double* x_all, double* g_all,
                         double* out_all, int n_scen, const int32_t* ids, int packed, double dx) {
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
    const size_t nb = g ? jb.size() / BT_COLS : (size_t)h.n_jac_main; /* the linear-row blocks: pair evaluations only */
    for (size_t b = 0; b < nb; b++) {
      const int32_t* bt = jb.data() + b * BT_COLS;
      memset(&store, 0xff, sizeof store);
      for (int phase = 0; phase < GJ_PHASES; phase++)
        for (int tid = 0; tid < GJ_THREADS; tid++) jac_block_phase<JR_ALL>(P, sid, bt, x, vals, g, tid, phase, sm);
    }
    for (int k = 0; k < h.n_vac; k++) dyn_noair_node(P, sid, x, vals, g, jac_node(P, h.vac_first + k));
  }
}

// packed: out_all is [n_scen][n_pack], else [n_scen][n_vals] from the template; g_all != NULL: pair evaluation.
extern "C" int emu_eval_central(const GelatoPlanDesc* d, const GelatoScenarioDesc* sc, const double* x_all, double* g_all,
                                double* out_all, int n_scen, const int32_t* ids, int packed, double step) {
  if (validate_desc(d) || !(step > 0.0)) return -1;
  PackedLayout L;
  build_packed_layout(d, L);
  std::vector<double> minus((size_t)n_scen * (size_t)L.n_pack);
  central_pass(d, sc, x_all, g_all, out_all, n_scen, ids, packed, step);
  central_pass(d, sc, x_all, nullptr, minus.data(), n_scen, ids, 1, -step);
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
