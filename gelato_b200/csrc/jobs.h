/* jobs.h -- the work items of the two fused kernels, as per-thread functions.
 *
 * A kernel block has a role (a row of the block table) and runs its job in phases separated by
 * block barriers.  Jacobian kernel (phases numbered 0, 2, 3; each role uses those it needs):
 *   phase 0  the expensive, shareable parts of the leaves: per air node 5 position items
 *            (pos_part) and 7 rotation items (rotq_part) cover all 14 finite-difference columns;
 *            vacuum nodes: 5 gravity items; the quaternion kinematics, one thread per node;
 *            event rows and fallback nodes: one full leaf per lane;
 *   phase 2  one thread per (node, column): the cheap per-column remainder on its own perturbed
 *            copy of the inputs, result parked in shared memory;
 *   phase 3  finite-difference quotients against the centre column, in the reference's operation
 *            order, scattered to their COO slots (lane-major: neighbouring threads, same formula).
 * Residual kernel: phase 0 position | rotation part (two threads per node), phase 1 the
 * right-hand sides, phase 2 D.X minus right-hand side for the 11 state columns.
 *
 * The functions are host+device so tests/emu can step through the same code on the CPU; the
 * shipped library only runs them inside CUDA kernels.
 *
 * Reference formulas: see the citations on each function; the perturbation protocol (which
 * inputs carry fl(fl(x+dx)-dx) residue when a given column is evaluated) is DESIGN.md "H3" /
 * SURVEY.md A.4.
 */
#ifndef GELATO_B200_JOBS_H_
#define GELATO_B200_JOBS_H_

#include "../../include/gelato_b200.h"
#include "physics.h"

/* ---- launch geometry (each overridable with -D for tuning experiments: tools/ab_probe.sh) ---------
 * One Jacobian block = 14 warps.  A block of 32 air nodes has 160 position items (5 full warps), 224
 * rotation items (7 full warps) and 32 quaternion items (1 warp): ONE long item per thread, every warp full;
 * the 14th warp computes the D.X products of a pair evaluation meanwhile.  Its 448 column items are one
 * round of the whole block.  A block of 32 aero rows in a pair evaluation carries a sixth position / eighth
 * rotation variant (the pristine state, for objfunc's row): 192 + 256 items = the 14 warps again.
 * (Measured against 8 warps x 32 nodes -- round 1: three rounds of rotation items on 3 warps --, 9 warps x 20
 * nodes, 7 warps x 16 nodes, 16 warps x 32 nodes: profiles/r02a_ab_probe.txt.)  Every item loop strides by
 * its thread-group size, so any geometry that satisfies the static_asserts is valid. */
#ifndef GJ_THREADS
#define GJ_THREADS 448   /* Jacobian kernel block */
#endif
#ifndef GJ_NODES
#define GJ_NODES 32      /* aero rows per Jacobian block */
#endif
#ifndef GD_NODES
#define GD_NODES 32      /* air dynamics nodes per Jacobian block */
#endif
#ifndef GJ_A_THREADS
#define GJ_A_THREADS 160 /* air dynamics blocks: threads [0, 160) position items; the rest rotation / quaternion / D.X items */
#endif
#ifndef GJA_A_THREADS
#define GJA_A_THREADS 192 /* aero blocks: threads [0, 192) position items; the rest rotation items */
#endif
#ifndef GD_GRAVITY_IN_POS
#define GD_GRAVITY_IN_POS 0 /* 1: the position items compute gravity too (round 1); 0: the quaternion items' warp does, which
                               shortens the longest chain of phase 0 (profiles/r02_ab_probe.txt) */
#endif
#ifndef GN_NODES
#define GN_NODES 32      /* no-air nodes per Jacobian block */
#endif
#ifndef GN_A_THREADS
#define GN_A_THREADS 160 /* no-air blocks: threads [0, 160) gravity items, the rest quaternion and D.X items */
#endif
/* Event jobs per Jacobian block, 16 lanes each.  Two jobs of different types in one warp run one after the other
 * (phase clocks: 69 000 cycles for the warp with an IIP and an antenna row against 37 000 for its neighbours), so
 * GJ_EVT_PER_WARP = 1 gives every job a warp of its own: the event block then takes 65 000 instead of 75 000 cycles
 * and a sens-only launch gains 1.5 %, but the timed pair evaluation (L2 flushed) loses 1 % on the same box
 * (profiles/r02h_ab_probe.txt) -- off. */
#ifndef GJ_EVT_PER_WARP
#define GJ_EVT_PER_WARP 0
#endif
#ifndef GJ_EVT
#define GJ_EVT (GJ_THREADS / (GJ_EVT_PER_WARP ? 32 : 16))
#endif
#ifndef GG_NODES
#define GG_NODES (GJ_THREADS / 16) /* nodes per block of the one-lane-per-column fallback (16 lanes each) */
#endif
#define GR_THREADS 128 /* residual kernel block */
#define GR_NODES 64    /* nodes per residual block */
#define NPV 5          /* distinct positions over the columns of one node */
#define NRV 7          /* distinct (position, time) pairs */
#define NPVA 6         /* aero rows: + the pristine position (objfunc's row in a pair evaluation) */
#define NRVA 8         /* aero rows: + the pristine (position, time) */
#define NQV 8          /* quaternion-kinematics variants: centre, q x4, u x2 (after the velocity pass), pristine */

static_assert(GJ_A_THREADS % 32 == 0 && GJ_A_THREADS < GJ_THREADS && GJ_THREADS % 32 == 0, "phase-0 thread groups are whole warps");
static_assert(GJA_A_THREADS % 32 == 0 && GJA_A_THREADS < GJ_THREADS, "phase-0 thread groups are whole warps");
static_assert(GN_A_THREADS % 32 == 0 && GN_A_THREADS < GJ_THREADS, "no-air thread groups are whole warps");
static_assert(GG_NODES * 16 <= GJ_THREADS && GJ_EVT * 16 <= GJ_THREADS, "lane maps");
#define GJ_MAX2(a, b) ((a) > (b) ? (a) : (b))
#define GJ_FQ_NODES GJ_MAX2(GJ_MAX2(GN_NODES, GD_NODES), GG_NODES) /* nodes the f and q arrays hold */
#define GJ_PR_NODES GJ_MAX2(GJ_NODES, GD_NODES)                    /* nodes (or aero rows) the pp and rq arrays hold */
static_assert(GJ_THREADS * 3 <= GJ_FQ_NODES * 14 * 3, "event jobs keep 3 values per thread in f");
static_assert(GN_NODES * NPV * 3 <= GJ_PR_NODES * NPVA * 8, "no-air gravity items fit the pp array");
static_assert(GR_THREADS == 2 * GR_NODES, "residual phase 0 uses two threads per node");

/* block roles */
enum { BR_DYN_AIR = 0, BR_DYN_NOAIR, BR_DYN_GEN, BR_AERO, BR_EVT, BR_LIN, BR_DYN /* residual kernel */ };
/* block table columns */
enum { BT_ROLE = 0, BT_JOB, BT_START, BT_COUNT, BT_COLS };
#define GJ_PHASES 4

struct PlanView {
  int S, N, M, n_vars, n_rows;
  long long n_vals;
  int payload_mode;
  int off_pos, off_vel, off_quat, off_u, off_t; /* offsets into x (mass at 0) */
  const int32_t* sec_i32;
  const int64_t* sec_i64;
  const double* sec_f64;
  long long sec_f64_sstride; /* per-scenario stride (0 = shared) */
  const double* d_pool;
  const double* tau_pool;
  const double* wind;
  long long wind_sstride;
  int n_wind;
  const double* ca;
  int n_ca;
  Units un;
  const double* unit_mass_scen; /* [n_scen] or NULL */
  int n_lin;
  const int32_t* lin_i32;
  const double* lin_f64;
  const double* lin_const_scen; /* [n_scen][n_lin] or NULL */
  int n_aero;
  const int32_t* aero_i32;
  const int64_t* aero_i64;
  const double* aero_f64;
  const uint8_t* rc_aero;
  int n_evt;
  const int32_t* evt_i32;
  const int64_t* evt_i64;
  const double* evt_f64;
  /* built by plan_host.h at plan creation */
  const struct NodeRec* node_rec; /* [N] collocation nodes in natural order */
  const struct NodeRec* jac_rec;  /* [N] the same records grouped by Jacobian block role */
  const struct AeroRec* aero_rows; /* [n_aero_rows] one record per aero constraint row */
  int n_aero_rows;
  /* packed output (plan_host.h: build_packed_layout): the Jacobian kernel writes only the INDEPENDENT
   * x-dependent values, contiguously per section, instead of the reference's COO slots */
  int packed;             /* 0: vals[n_vals] in COO order | 1: packed[n_pack] */
  long long n_pack;
  const int64_t* sec_pk;  /* [S][GS_I64_COLS] offsets into the packed vector */
  const int64_t* aero_pk; /* [n_aero][GA_I64_COLS] */
  const int64_t* evt_pk;  /* [n_evt][GE_I64_COLS] */
};

/* working arrays of one Jacobian block: shared memory in the kernel (JacStore, 46 KB), a plain struct
 * in the host emulator; the jobs reach them through the pointers of JacScratch. */
#define GJ_PP_LEN (GJ_PR_NODES * NPVA * PP_COLS) /* pos_part per (node, position variant); no-air: gravity[3] */
#define GJ_RQ_LEN (GJ_PR_NODES * NRVA * RQ_COLS) /* rotq_part per (node, rotation variant) */
#define GJ_LH_LEN (GJ_FQ_NODES * 11)             /* D.X per (node, state column): position 3 | quaternion 4 | velocity 3 | mass */
#define GJ_F_LEN (GJ_FQ_NODES * 14 * 3)         /* leaf value per (node, column lane); events: per thread */
#define GJ_Q_LEN (GJ_FQ_NODES * NQV * 4)        /* quaternion kinematics per (node, variant) */
struct JacStore {
  double pp[GJ_PP_LEN];
  double rq[GJ_RQ_LEN];
  double q[GJ_Q_LEN];
  double f[GJ_F_LEN];
  double lh[GJ_LH_LEN];
};
struct JacScratch {
  double* pp;
  double* rq;
  double* q;
  double* f;
  double* lh;
};
P_HD JacScratch jac_scratch(JacStore& st) {
  JacScratch sm;
  sm.pp = st.pp; sm.rq = st.rq; sm.q = st.q; sm.f = st.f; sm.lh = st.lh;
  return sm;
}
/* shared memory of one residual block */
struct ResScratch {
  double f[GR_NODES][3];
  double q[GR_NODES][4];
  double pp[GR_NODES][PP_COLS];
  double rq[GR_NODES][RQ_COLS];
};

/* fl(fl(x + dx) - dx): what a perturb/restore cycle leaves behind */
P_HD double residue(double x, double dx) {
  double y = x + dx;
  return y - dx;
}
/* n perturb/restore cycles.  n is a small per-variable count compiled into the plan (how many earlier
 * groups of `sens` touched the variable); four predicated steps cover it without a data-dependent
 * branch (ncu r01j: the loop form was 16 % of the instruction-fetch stalls), a loop takes any excess. */
P_HD double residue_n(double x, double dx, int n) {
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const double y = residue(x, dx);
    x = (i < n) ? y : x;
  }
  for (int i = 4; i < n; i++) x = residue(x, dx);
  return x;
}

/* num / dx for the finite-difference quotients (the plan's dx > 0, checked at plan creation; the -h pass of
 * central differences runs with dx < 0).  Many quotients have an exactly zero numerator (a column that does not
 * move an output); IEEE gives 0/dx = 0 with the numerator's sign for dx > 0, and saying so skips the division's
 * slow path, which the GPU's software FP64 division takes for zero numerators (ncu r01b: 8 % of all instructions).
 * For dx < 0 the zero keeps the numerator's sign too, unlike IEEE's 0/dx: DESIGN.md H6 makes that the rule. */
P_HD double fd_div(double num, double dx) { return num == 0.0 ? num : gm_div(num, dx); }
/* the same with the reciprocal of dx computed once by the caller (gmath.h: gm_div_by is the IEEE quotient) */
P_HD double fd_div_by(double num, const GmRcp Rdx) { return num == 0.0 ? num : gm_div_by(num, Rdx); }
/* a central-difference value from the forward protocol's values with steps +h and -h (DESIGN.md H6) */
P_HD double fd_central(double q_plus, double q_minus) { return (q_plus + q_minus) * 0.5; }

P_HD Units scen_units(const PlanView& P, int scen) {
  Units u = P.un;
  if (P.unit_mass_scen) u.mass = P.unit_mass_scen[scen];
  return u;
}
P_HD SecParam sec_param(const PlanView& P, int scen, int sec) {
  const double* f = P.sec_f64 + (long long)scen * P.sec_f64_sstride + (long long)sec * GS_F64_COLS;
  SecParam sp;
  sp.thrust = f[GS_THRUST];
  sp.massflow = f[GS_MASSFLOW];
  sp.ref_area = f[GS_REF_AREA];
  sp.nozzle_area = f[GS_NOZZLE_AREA];
  return sp;
}
P_HD Tables scen_tables(const PlanView& P, int scen) {
  Tables tb;
  tb.wind = P.wind + (long long)scen * P.wind_sstride;
  tb.n_wind = P.n_wind;
  tb.ca = P.ca;
  tb.n_ca = P.n_ca;
  return tb;
}

/* PSparams.time_nodes (SectionParameters.py:77-81): row 0 = to, row r>=1 = LGR point r-1 */
P_HD double time_node(const double* tau, int r, double to, double tf) {
  if (r == 0) return to;
  return tau[r - 1] * (tf - to) / 2 + (tf + to) / 2;
}

/* ========================================================================= */
/* Dynamics: what each finite-difference column of a node sees                */
/*   column lanes: 0 centre | 1 mass | 2-4 position | 5-7 velocity |          */
/*                 8-11 quaternion | 12 to | 13 tf | 14 dyn_pos entries       */
/*   lanes 0-6 also name the quaternion-kinematics variants (centre, q x4,    */
/*   u x2)                                                                    */
/* reference: con_dynamics.py:292-496 (velocity), :536-632 (quaternion),      */
/*            :155-213 (position)                                             */
/* ========================================================================= */
/* everything a job needs to know about one collocation node, in one 32-byte record (two 16-byte loads)
 * instead of a chain of dependent table look-ups; built by plan_host.h */
struct alignas(16) NodeRec {
  int32_t sec, j, row, ua; /* section, LGR node index inside it, state row, first control row of the section */
  int32_t n, flags, d_off, tau_off; /* nodes in the section, GSF_*, offsets of its D block and tau */
};
struct NodeRef {
  int sec, j, row, ua, n, flags, d_off, tau_off;
  const int32_t* si; /* the section's row of sec_i32 (address only: no load) */
};
P_HD NodeRef node_from_rec(const PlanView& P, const NodeRec& q) {
  NodeRef r;
  r.sec = q.sec; r.j = q.j; r.row = q.row; r.ua = q.ua;
  r.n = q.n; r.flags = q.flags; r.d_off = q.d_off; r.tau_off = q.tau_off;
  r.si = P.sec_i32 + q.sec * GS_I32_COLS;
  return r;
}
/* the same for one aero constraint row */
struct alignas(16) AeroRec {
  int32_t job, r, sec, row;        /* aero job, row inside it, section, state row */
  int32_t kind, nk, tau_off, row0; /* 0 alpha / 1 q / 2 q-alpha, rows of the job, tau offset, first residual row */
};

/* node k of the Jacobian kernel's role-grouped order / node g of the natural order */
P_HD NodeRef jac_node(const PlanView& P, int k) { return node_from_rec(P, P.jac_rec[k]); }
P_HD NodeRef res_node(const PlanView& P, int g) { return node_from_rec(P, P.node_rec[g]); }

/* mass, pos[3], vel[3], quat[4] of state row `row` as column `lane` evaluates them: the
 * reference perturbs views of xdict in place, so variables visited before this column
 * carry fl(fl(x+dx)-dx) and the column's own variable carries x+dx (SURVEY.md A.4) */
P_HD void dyn_col_state(const PlanView& P, const double* x, int row, int lane, bool air_fd, double dx, double* v) {
  v[0] = x[row];
  for (int k = 0; k < 3; k++) v[1 + k] = x[P.off_pos + 3 * row + k];
  for (int k = 0; k < 3; k++) v[4 + k] = x[P.off_vel + 3 * row + k];
  for (int k = 0; k < 4; k++) v[7 + k] = x[P.off_quat + 4 * row + k];
  if (lane == 0) return;
  const int pidx = (lane <= 11) ? lane - 1 : 11;
#pragma unroll
  for (int w = 0; w < 11; w++) {
    const bool in_protocol = (w < 4) || (w >= 7) || air_fd; /* velocity columns exist for air sections only */
    if (!in_protocol) continue;
    if (w < pidx) v[w] = residue(v[w], dx);
    else if (w == pidx) v[w] = v[w] + dx;
  }
}

/* The 14 columns see only NPV = 5 distinct positions and NRV = 7 distinct (position,
 * node time) pairs:
 *   pv 0 pristine (lanes 0,1) | 1-3 axis pv-1 perturbed (lanes 2-4) | 4 all restored (lanes 5-13)
 *   rv 0-4 = pv 0-4 at the nominal node time | 5 = pv 4, to+dx (lane 12) | 6 = pv 4, tf+dx (lane 13) */
P_HD int lane_pv(int lane) { return lane < 2 ? 0 : (lane <= 4 ? lane - 1 : 4); }
P_HD int lane_rv(int lane) { return lane < 2 ? 0 : (lane <= 4 ? lane - 1 : (lane <= 11 ? 4 : lane - 7)); }
P_HD int rv_pv(int rv) { return rv < 4 ? rv : 4; }

/* non-dimensional position variant pv of a base position b[3] */
P_HD void pos_variant(const double* b, int pv, double dx, double* out) {
  for (int k = 0; k < 3; k++) {
    double p = b[k];
    if (pv == 4 || (pv >= 1 && k < pv - 1)) p = residue(p, dx);
    else if (pv >= 1 && k == pv - 1) p = p + dx;
    out[k] = p;
  }
}

/* quaternion kinematics (con_dynamics.py:580-613): the state already carries one residue from
 * the velocity pass; variants 0 centre | 1-4 quaternion component | 5-6 control | 7 the PRISTINE state
 * (what objfunc evaluates, con_dynamics.py:525-530: the residual rows of a pair evaluation) */
P_HD void dyn_quat_variant(const PlanView& P, const double* x, const NodeRef& nr, const Units& un, int var, double* out) {
  const double dx = un.dx;
  double qv[4], uv[2];
  for (int k = 0; k < 4; k++) qv[k] = x[P.off_quat + 4 * nr.row + k];
  for (int k = 0; k < 2; k++) uv[k] = x[P.off_u + 2 * (nr.ua + nr.j) + k];
  if (var != 7)
    for (int k = 0; k < 4; k++) qv[k] = residue(qv[k], dx);
  if (var >= 1 && var <= 4) {
    const int k = var - 1;
    for (int w = 0; w < 4; w++) {
      if (w < k) qv[w] = residue(qv[w], dx);
      else if (w == k) qv[w] = qv[w] + dx;
    }
  } else if (var == 5 || var == 6) {
    const int k = var - 5;
    for (int w = 0; w < 4; w++) qv[w] = residue(qv[w], dx);
    for (int w = 0; w < 2; w++) {
      if (w < k) uv[w] = residue(uv[w], dx);
      else if (w == k) uv[w] = uv[w] + dx;
    }
  }
  Quat d = rhs_quaternion(q4(qv[0], qv[1], qv[2], qv[3]), uv[0], uv[1], un.u);
  out[0] = d.w;
  out[1] = d.x;
  out[2] = d.y;
  out[3] = d.z;
}
P_HD void dyn_quat_variants(const PlanView& P, const double* x, const NodeRef& nr, const Units& un, double* out) {
  for (int var = 0; var < NQV; var++) dyn_quat_variant(P, x, nr, un, var, out + 4 * var);
}

/* finite-difference quotients of one (node, lane) and their output slots.
 * fc / fl: velocity right-hand side at the centre / in this lane; qc / ql: quaternion
 * kinematics at the centre / in variant `lane`.
 * COO output (P.packed == 0): the reference's slots.  Packed output: the same values, but only the
 * independent ones, contiguous per section -- the node-diagonal entries of the dense D (x) I blocks become
 * dense [9][n] / [4n][4] arrays, the `tf` halves that are exact negations of the `to` halves and the 3n
 * identical entries of eqcon_dyn_pos / velocity are not written (plan_host.h: build_packed_layout lists which
 * COO slot is which packed value, with what sign). */
P_HD void dyn_scatter(const PlanView& P, int scen, const double* x, double* vals, const NodeRef& nr, int lane,
                      const double* fc, const double* fl, const double* qc, const double* ql) {
  const bool pk = P.packed != 0;
  const int64_t* sj = (pk ? P.sec_pk : P.sec_i64) + nr.sec * GS_I64_COLS;
  const int n = nr.n, j = nr.j, row = nr.row;
  const Units un = scen_units(P, scen);
  const double dx = un.dx, ut = un.t;
  const GmRcp Rdx = gm_rcp(dx);
  const bool air_fd = nr.flags & GSF_AIR_FD, hold = nr.flags & GSF_HOLD;
  const double to = x[P.off_t + nr.sec], tf = x[P.off_t + nr.sec + 1];
  const double dt = tf - to;
  const long long n3 = 3LL * n, n4 = 4LL * n, nn1 = (long long)n * (n + 1);

  /* ---- velocity dynamics: -(f_p - f_c)/dx*(tf-to)*unit_t/2 (con_dynamics.py:372) ---- */
  if (lane >= 1 && lane <= 11 && !(lane >= 5 && lane <= 7 && !air_fd)) {
    double rh[3];
    for (int k = 0; k < 3; k++) rh[k] = fd_div_by(-(fl[k] - fc[k]), Rdx) * dt * ut / 2.0;
    if (lane == 1) {
      for (int k = 0; k < 3; k++) vals[sj[GS_JV_MASS] + 3LL * j + k] = rh[k];
    } else if (lane <= 4) {
      const int kk = lane - 2;
      for (int k = 0; k < 3; k++) vals[sj[GS_JV_POS] + kk * n3 + 3LL * j + k] = rh[k];
    } else if (lane <= 7) {
      const int kk = lane - 5; /* submat_vel[3j+ki, 3(j+1)+kk] += rh[ki]  (:415-416) */
      const double d_diag = P.d_pool[nr.d_off + (long long)j * (n + 1) + (j + 1)];
      for (int ki = 0; ki < 3; ki++) {
        const double base = (ki == kk) ? d_diag : 0.0;
        const long long at = pk ? (long long)(ki * 3 + kk) * n + j : (ki * 3 + kk) * nn1 + (long long)j * (n + 1) + (j + 1);
        vals[sj[GS_JV_VEL] + at] = base + rh[ki];
      }
    } else {
      const int kk = lane - 8;
      for (int k = 0; k < 3; k++) vals[sj[GS_JV_QUAT] + kk * n3 + 3LL * j + k] = rh[k];
    }
  }
  if (lane == 12) {
    if (air_fd) { /* :454-465 */
      const double to_p = to + dx;
      for (int k = 0; k < 3; k++)
        vals[sj[GS_JV_T] + 3LL * j + k] = fd_div_by(-(fl[k] * (tf - to_p) - fc[k] * dt), Rdx) * ut / 2.0;
    } else { /* :478-480 */
      for (int k = 0; k < 3; k++) {
        const double rh_to = fc[k] * ut / 2.0;
        vals[sj[GS_JV_T] + 3LL * j + k] = rh_to;
        if (!pk) vals[sj[GS_JV_T] + n3 + 3LL * j + k] = -rh_to;
      }
    }
  }
  if (lane == 13 && air_fd) { /* :466-477 */
    const double tf_p = tf + dx;
    for (int k = 0; k < 3; k++)
      vals[sj[GS_JV_T] + n3 + 3LL * j + k] = fd_div_by(-(fl[k] * (tf_p - to) - fc[k] * dt), Rdx) * ut / 2.0;
  }
  /* ---- position dynamics (analytic, depends on x through vel and t): :180-195 ---- */
  if (lane == 14) {
    const GmRcp Rp = gm_rcp(un.pos);
    const double rh_vel = gm_div_by(-un.vel * dt * ut / 2.0, Rp);
    if (pk) {
      if (j == 0) vals[sj[GS_JP_VEL]] = rh_vel; /* one value per section */
    } else {
      for (int k = 0; k < 3; k++) vals[sj[GS_JP_VEL] + 3LL * j + k] = rh_vel;
    }
    for (int k = 0; k < 3; k++) {
      const double rh_to = gm_div_by(x[P.off_vel + 3 * row + k] * un.vel * ut / 2.0, Rp);
      vals[sj[GS_JP_T] + 3LL * j + k] = rh_to;
      if (!pk) vals[sj[GS_JP_T] + n3 + 3LL * j + k] = -rh_to;
    }
  }
  /* ---- quaternion kinematics: :580-625 ---- */
  if (!hold) {
    if (lane >= 1 && lane <= 6) {
      double rh[4];
      for (int a = 0; a < 4; a++) rh[a] = fd_div_by(-(ql[a] - qc[a]), Rdx) * dt * ut / 2.0;
      if (lane <= 4) {
        const int kk = lane - 1; /* submat_quat[4j+a, 4(j+1)+kk] += rh[a] */
        const double d_diag = P.d_pool[nr.d_off + (long long)j * (n + 1) + (j + 1)];
        for (int a = 0; a < 4; a++) {
          const double base = (a == kk) ? d_diag : 0.0;
          const long long at = pk ? (4LL * j + a) * 4 + kk : (4LL * j + a) * (4LL * (n + 1)) + 4LL * (j + 1) + kk;
          vals[sj[GS_JQ_QUAT] + at] = base + rh[a];
        }
      } else {
        const int kk = lane - 5;
        for (int a = 0; a < 4; a++) vals[sj[GS_JQ_U] + kk * n4 + 4LL * j + a] = rh[a];
      }
    } else if (lane == 0) {
      for (int a = 0; a < 4; a++) {
        const double rh_to = qc[a] * ut / 2.0;
        vals[sj[GS_JQ_T] + 4LL * j + a] = rh_to;
        if (!pk) vals[sj[GS_JQ_T] + n4 + 4LL * j + a] = -rh_to;
      }
    }
  }
}

P_HD void dyn_lh_item(const PlanView& P, const double* x, const NodeRef& nr, int grp, double* lh);
P_HD void dyn_lh_vel_col(const PlanView& P, const double* x, const NodeRef& nr, int k, double* lh);
P_HD void dyn_res_finish(const PlanView& P, int scen, const double* x, double* g, const NodeRef& nr, int grp,
                         const double* lh, const double* f3, const double* q4v);

/* pair evaluation, phase 0: the D.X products of the block's nodes, by the threads the long items leave idle
 * (`idx` of `n_group` threads, the first `n_busy` of which have a long item): hidden behind pos_part / rotq_part */
P_HD void dyn_lh_block(const PlanView& P, const double* x, int start, int count, int idx, int n_group, int n_busy,
                       const JacScratch& sm) {
  const int spare = n_group - n_busy;
  int first = idx, step = n_group;
  if (spare > 0) {
    if (idx < n_busy) return;
    first = idx - n_busy;
    step = spare;
  }
  for (int item = first; item < count * 4; item += step) {
    const int grp = item / count, nl = item - grp * count;
    dyn_lh_item(P, x, jac_node(P, start + nl), grp, sm.lh + nl * 11);
  }
}
/* The same products for the air-node blocks, spread by measured slack (tools/phase_clocks.py: with all of them on
 * the one spare warp that warp ended phase 0 last, 17 000 cycles against 15 200 for the position items and 12 800 for
 * the rotation items): the spare warp takes the position and quaternion products of its lane's node, the first
 * four rotation warps add ONE column each after their item -- velocity x, y, z and mass.  Needs a whole spare warp
 * and four busy ones; other geometries keep dyn_lh_block. */
P_HD void dyn_lh_spread(const PlanView& P, const double* x, int start, int count, int idx, int n_busy, const JacScratch& sm) {
  if (idx >= n_busy) {
    const int nl = idx - n_busy;
    if (nl < count) {
      const NodeRef nr = jac_node(P, start + nl);
      dyn_lh_item(P, x, nr, 0, sm.lh + nl * 11);
      dyn_lh_item(P, x, nr, 1, sm.lh + nl * 11);
    }
    return;
  }
  const int col = idx >> 5, nl = idx & 31;
  if (col >= 4 || nl >= count) return;
  const NodeRef nr = jac_node(P, start + nl);
  if (col == 3) dyn_lh_item(P, x, nr, 3, sm.lh + nl * 11);
  else dyn_lh_vel_col(P, x, nr, col, sm.lh + nl * 11);
}

/* all 15 lanes of the nodes of a block, leaf values laid out f[(nl*14 + lane)*3], q[(nl*NQV + var)*4];
 * with g != NULL (pair evaluation) also the collocation defects of the same nodes: the D.X of phase 0 minus
 * the centre column's right-hand side (pristine x) / the pristine quaternion variant -- objfunc's rows without
 * a second pass over the physics */
P_HD void dyn_scatter_block(const PlanView& P, int scen, const double* x, double* vals, double* g, int start, int count,
                            int tid, int nthreads, const JacScratch& sm) {
  /* lane-major items: neighbouring threads run the same column's formula on neighbouring nodes */
  for (int item = tid; item < count * 15; item += nthreads) {
    const int lane = item / count, nl = item - lane * count;
    const NodeRef nr = jac_node(P, start + nl);
    const double* fc = sm.f + (nl * 14) * 3;
    const double* qc = sm.q + (nl * NQV) * 4;
    dyn_scatter(P, scen, x, vals, nr, lane, fc, fc + (lane < 14 ? lane : 0) * 3, qc, qc + (lane < 7 ? lane : 0) * 4);
  }
  if (g) {
    /* the threads the last scatter round leaves idle go first */
    for (int item = nthreads - 1 - tid; item < count * 4; item += nthreads) {
      const int grp = item / count, nl = item - grp * count;
      const NodeRef nr = jac_node(P, start + nl);
      dyn_res_finish(P, scen, x, g, nr, grp, sm.lh + nl * 11, sm.f + (nl * 14) * 3, sm.q + (nl * NQV + 7) * 4);
    }
  }
}

/* ========================================================================= */
/* Jacobian kernel, DYN_AIR role: GD_NODES air nodes per block                 */
/*   0  threads [0, GJ_A_THREADS): position items (node, pv) -> pos_part;      */
/*      the others: rotation items (node, rv) -> rotq_part, then one           */
/*      quaternion item per node (the NQV kinematics variants)                 */
/*   2  column items (node, lane 0-13): wind into ECI axes, per-column         */
/*      remainder                                                             */
/*   3  finite-difference quotients -> output slots (+ defects, pair mode)     */
/*   (phase 1 is unused: the numbering is shared with the other roles)        */
/* ========================================================================= */
GM_HD_INL void dyn_air_phase(const PlanView& P, int scen, const double* x, double* vals, double* g, int start, int count,
                        int tid, int phase, const JacScratch& sm) {
  const Units un = scen_units(P, scen);
  const double dx = un.dx;
  if (phase == 0) {
    if (tid < GJ_A_THREADS) {
      const Tables tb = scen_tables(P, scen);
      for (int item = tid; item < count * NPV; item += GJ_A_THREADS) {
        const int nl = item / NPV, pv = item - nl * NPV;
        const NodeRef nr = jac_node(P, start + nl);
        double p[3];
        pos_variant(x + P.off_pos + 3 * nr.row, pv, dx, p);
        /* gravity is independent of the geodetic / atmosphere chain: the quaternion items' warp computes it */
        pos_part(p[0] * un.pos, p[1] * un.pos, p[2] * un.pos, tb.wind, tb.n_wind, GD_GRAVITY_IN_POS ? (PW_GRAVITY | PW_SOUND) : PW_SOUND,
                 sm.pp + (nl * NPV + pv) * PP_COLS);
      }
      return;
    }
    /* rotation items first (whole warps of them), then one quaternion item per node; the threads left over
     * compute the D.X products of a pair evaluation */
    const int nb = GJ_THREADS - GJ_A_THREADS, idx = tid - GJ_A_THREADS;
    for (int item = idx; item < count * (NRV + 1); item += nb) {
      if (item >= count * NRV) {
        const int qn = item - count * NRV;
        const NodeRef nr = jac_node(P, start + qn);
        if (!(nr.flags & GSF_HOLD)) dyn_quat_variants(P, x, nr, un, sm.q + qn * NQV * 4);
        if (!GD_GRAVITY_IN_POS) { /* the node's five gravity vectors: ~300 instructions each, next to ~500 for the variants */
          for (int pv = 0; pv < NPV; pv++) {
            double p[3];
            pos_variant(x + P.off_pos + 3 * nr.row, pv, dx, p);
            const Vec3 gr = gravity_eci(v3(p[0] * un.pos, p[1] * un.pos, p[2] * un.pos));
            double* o = sm.pp + (qn * NPV + pv) * PP_COLS;
            o[PP_GX] = gr.x;
            o[PP_GY] = gr.y;
            o[PP_GZ] = gr.z;
          }
        }
        continue;
      }
      const int nl = item / NRV, rv = item - nl * NRV;
      const NodeRef nr = jac_node(P, start + nl);
      double p[3];
      pos_variant(x + P.off_pos + 3 * nr.row, rv_pv(rv), dx, p);
      const double to0 = x[P.off_t + nr.sec], tf0 = x[P.off_t + nr.sec + 1];
      const double to = (rv == 5) ? to0 + dx : to0;
      const double tf = (rv == 6) ? tf0 + dx : tf0;
      const double tn = time_node(P.tau_pool + nr.tau_off, nr.j + 1, to, tf);
      rotq_part(p[0] * un.pos, p[1] * un.pos, p[2] * un.pos, tn, sm.rq + (nl * NRV + rv) * RQ_COLS);
    }
    if (g) {
      if (GD_NODES == 32 && nb - GD_NODES * (NRV + 1) >= 32) dyn_lh_spread(P, x, start, count, idx, GD_NODES * (NRV + 1), sm);
      else dyn_lh_block(P, x, start, count, idx, nb, count * (NRV + 1), sm);
    }
  } else if (phase == 2) {
    for (int item = tid; item < count * 14; item += GJ_THREADS) {
      const int nl = item / 14, lane = item - nl * 14;
      const NodeRef nr = jac_node(P, start + nl);
      double v[11], rp[RP_COLS];
      dyn_col_state(P, x, nr.row, lane, true, dx, v);
      const double* pp = sm.pp + (nl * NPV + lane_pv(lane)) * PP_COLS;
      /* the wind of this column's position, turned into ECI axes with this column's (position, time)
       * quaternion: 56 flops, cheaper to repeat per column than a block barrier for 7 items per node */
      rot_wind(sm.rq + (nl * NRV + lane_rv(lane)) * RQ_COLS, pp[PP_WIND_N], pp[PP_WIND_E], rp);
      const Vec3 f = rhs_velocity_air_col(v[0], v3(v[1], v[2], v[3]), v3(v[4], v[5], v[6]), q4(v[7], v[8], v[9], v[10]),
                                          pp, rp, sec_param(P, scen, nr.sec), un, scen_tables(P, scen));
      double* o = sm.f + (nl * 14 + lane) * 3;
      o[0] = f.x;
      o[1] = f.y;
      o[2] = f.z;
    }
  } else {
    dyn_scatter_block(P, scen, x, vals, g, start, count, tid, GJ_THREADS, sm);
  }
}

/* ========================================================================= */
/* Jacobian kernel, DYN_NOAIR role: GN_NODES vacuum nodes per block           */
/*   0  gravity items (node, pv) | quaternion kinematics                      */
/*   2  column items (node, 9 lanes: centre, mass, position x3, quaternion x4)*/
/*   3  quotients -> output slots (+ defects, pair mode)                      */
/* ========================================================================= */
GM_HD_INL void dyn_noair_phase(const PlanView& P, int scen, const double* x, double* vals, double* g, int start, int count,
                          int tid, int phase, const JacScratch& sm) {
  const Units un = scen_units(P, scen);
  const double dx = un.dx;
  if (phase == 0) {
    if (tid < GN_A_THREADS) {
      for (int item = tid; item < count * NPV; item += GN_A_THREADS) {
        const int nl = item / NPV, pv = item - nl * NPV;
        const NodeRef nr = jac_node(P, start + nl);
        double p[3];
        pos_variant(x + P.off_pos + 3 * nr.row, pv, dx, p);
        const Vec3 gr = gravity_eci(v3(p[0] * un.pos, p[1] * un.pos, p[2] * un.pos));
        double* o = sm.pp + (nl * NPV + pv) * 3;
        o[0] = gr.x;
        o[1] = gr.y;
        o[2] = gr.z;
      }
    } else {
      const int nb = GJ_THREADS - GN_A_THREADS, idx = tid - GN_A_THREADS;
      for (int qn = idx; qn < count; qn += nb) {
        const NodeRef nr = jac_node(P, start + qn);
        if (!(nr.flags & GSF_HOLD)) dyn_quat_variants(P, x, nr, un, sm.q + qn * NQV * 4);
      }
      if (g) dyn_lh_block(P, x, start, count, idx, nb, count, sm);
    }
  } else if (phase == 2) {
    for (int item = tid; item < count * 9; item += GJ_THREADS) {
      const int nl = item / 9, c9 = item - nl * 9;
      const int lane = c9 < 5 ? c9 : c9 + 3;
      const NodeRef nr = jac_node(P, start + nl);
      double v[11];
      dyn_col_state(P, x, nr.row, lane, false, dx, v);
      const double* gr = sm.pp + (nl * NPV + lane_pv(lane)) * 3;
      const Vec3 f = rhs_velocity_noair_col(v[0], q4(v[7], v[8], v[9], v[10]), v3(gr[0], gr[1], gr[2]),
                                            sec_param(P, scen, nr.sec), un);
      double* o = sm.f + (nl * 14 + lane) * 3;
      o[0] = f.x;
      o[1] = f.y;
      o[2] = f.z;
    }
  } else if (phase == 3) {
    dyn_scatter_block(P, scen, x, vals, g, start, count, tid, GJ_THREADS, sm);
  }
}

/* ========================================================================= */
/* Vacuum nodes, ONE THREAD PER NODE (kernel k_jacobian_noair): a vacuum        */
/* right-hand side is ~70 flops, so sharing gravity among its columns through   */
/* shared memory and two block barriers cost more than it saved -- the blocks   */
/* were latency bound with most threads idle (ncu r02b: 0.084 ms for 2 % of the */
/* arithmetic).  Here a thread walks its share of a node's columns in registers */
/* and stores each quotient as soon as it has it; one barrier (after the values */
/* a node's threads share are staged) and enough resident threads to hide the  */
/* chain.  Same per-(node, lane) formulas, same bits.                          */
/* ========================================================================= */
/* One node's columns in GV_PARTS independent parts (a warp per part in k_jacobian_noair: the parts differ in code
 * path, so they must not share a warp).  Every value is a pure function of (node, lane): each part recomputes the
 * centre column it differences against (cheap once gravity is shared) and the dependent chain is 3x shorter.
 *   part 0: lane 0 (the analytic t columns), lanes 1, 2      part 2: lanes 6, 8, 9
 *   part 1: lanes 3, 4, 5                                    part 3: lanes 10, 11
 * and, in a pair evaluation, the node's defect rows: velocity with part 1, position with part 2, quaternion and mass
 * with part 3.  Lanes 5-7 carry no velocity columns in vacuum (5, 6: the u columns of the quaternion rows; 7: nothing).
 * (The defects as a fifth part, 160-thread blocks, measured slower: 0.075 against 0.062 ms.)
 * The J2 gravity vector -- the expensive piece of a vacuum column -- has only NPV = 5 distinct arguments per node
 * (pristine, x / y / z perturbed, all restored); the parts would evaluate 10 of them between themselves.  Phase A
 * (dyn_noair_stage, one variant per warp, the first warp two) puts the five into shared memory, phase B
 * (dyn_noair_part) reads them.  Phase A also stages what every part reads of the node -- its pristine mass,
 * quaternion, velocity and controls, the section's times, thrust and output offsets -- so that phase B loads none
 * of it from global memory, where every output store before a load would force that load to be issued again. */
#define GV_PARTS 4
struct NoairStage {
  double m, q[4], u[2], vel[3], to, tf, thrust;
  double grav[NPV * 3]; /* [pv][3] */
  int64_t sj[GS_I64_COLS]; /* the section's row of sec_pk (packed output) or sec_i64 (COO) */
  double pad; /* an odd number of 8-byte words: an array of these, one per lane, is free of shared-memory bank conflicts */
};
static_assert(sizeof(NoairStage) % 16 == 8, "NoairStage: odd number of 8-byte words");

/* phase A, warp `part`: its share of the node's stage */
P_HD void dyn_noair_stage(const PlanView& P, int scen, const double* x, const NodeRef& nr, int part, NoairStage& s) {
  const Units un = scen_units(P, scen);
  const int row = nr.row;
  for (int pv = part; pv < NPV; pv += GV_PARTS) {
    double p[3];
    pos_variant(x + P.off_pos + 3 * row, pv, un.dx, p);
    const Vec3 gr = gravity_eci(v3(p[0] * un.pos, p[1] * un.pos, p[2] * un.pos));
    s.grav[3 * pv] = gr.x; s.grav[3 * pv + 1] = gr.y; s.grav[3 * pv + 2] = gr.z;
  }
  if (part == 1) {
    s.m = x[row];
    for (int k = 0; k < 4; k++) s.q[k] = x[P.off_quat + 4 * row + k];
    for (int k = 0; k < 2; k++) s.u[k] = (nr.flags & GSF_HOLD) ? 0.0 : x[P.off_u + 2 * (nr.ua + nr.j) + k];
  } else if (part == 2) {
    for (int k = 0; k < 3; k++) s.vel[k] = x[P.off_vel + 3 * row + k];
    s.to = x[P.off_t + nr.sec];
    s.tf = x[P.off_t + nr.sec + 1];
  } else if (part == 3) {
    s.thrust = sec_param(P, scen, nr.sec).thrust;
    const int64_t* sj = (P.packed ? P.sec_pk : P.sec_i64) + nr.sec * GS_I64_COLS;
    for (int c = 0; c < GS_I64_COLS; c++) s.sj[c] = sj[c];
  }
}

/* gm_div_by, with the zero numerator answered directly: a signed zero over a normal d is the zero with the sign
 * a / d has.  The coast arcs' thrust is zero, and the division routine reaches that quotient only through its slow
 * path.  Same bits as a / d. */
P_HD double noair_div_by(double a, const GmRcp R) {
  if (a == 0.0 && R.ok) return gm_u2d((gm_d2u(a) ^ gm_d2u(R.d)) & GM_SIGN_MASK);
  return gm_div_by(a, R);
}
/* vacuum column `lane`: rhs_velocity_noair_col on the mass and quaternion dyn_col_state gives the lane and on the
 * staged gravity of its position; Rv = gm_rcp(un.vel), shared by every column */
P_HD void noair_col(const NoairStage& s, int lane, const Units& un, const GmRcp Rv, double* f) {
  const double dx = un.dx;
  double m = s.m;
  if (lane == 1) m = m + dx;
  else if (lane >= 2) m = residue(m, dx);
  const int pidx = lane <= 11 ? lane - 1 : 11;
  double q[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    double a = s.q[k];
    if (lane != 0) {
      if (7 + k < pidx) a = residue(a, dx);
      else if (7 + k == pidx) a = a + dx;
    }
    q[k] = a;
  }
  const double mass = m * un.mass;
  const Vec3 tdir = quatrot(quatconj(q4(q[0], q[1], q[2], q[3])), v3(1.0, 0.0, 0.0));
  const Vec3 thr = scale3(s.thrust, tdir);
  const GmRcp Rm = gm_rcp(mass);
  const double* gv = s.grav + 3 * lane_pv(lane);
  f[0] = noair_div_by(noair_div_by(thr.x, Rm) + gv[0], Rv);
  f[1] = noair_div_by(noair_div_by(thr.y, Rm) + gv[1], Rv);
  f[2] = noair_div_by(noair_div_by(thr.z, Rm) + gv[2], Rv);
}
/* dyn_quat_variant on the staged quaternion and controls, every index a constant (the variant is a loop variable
 * of dyn_noair_part: indexing by it put qv / uv on the stack) */
P_HD void noair_quat_variant(const NoairStage& s, int var, const Units& un, double* out) {
  const double dx = un.dx;
  double qv[4], uv[2];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    double a = s.q[k];
    if (var != 7) a = residue(a, dx);
    if (var >= 1 && var <= 4) {
      if (k < var - 1) a = residue(a, dx);
      else if (k == var - 1) a = a + dx;
    } else if (var == 5 || var == 6) {
      a = residue(a, dx);
    }
    qv[k] = a;
  }
#pragma unroll
  for (int k = 0; k < 2; k++) {
    double b = s.u[k];
    if (var == 5 || var == 6) {
      if (k < var - 5) b = residue(b, dx);
      else if (k == var - 5) b = b + dx;
    }
    uv[k] = b;
  }
  const Quat d = rhs_quaternion(q4(qv[0], qv[1], qv[2], qv[3]), uv[0], uv[1], un.u);
  out[0] = d.w; out[1] = d.x; out[2] = d.y; out[3] = d.z;
}
/* dyn_scatter for a vacuum node (no velocity / time finite differences), on the staged values; Rdx = gm_rcp(un.dx) */
P_HD void dyn_noair_scatter(const PlanView& P, double* vals, const NodeRef& nr, const NoairStage& s, const Units& un,
                            const GmRcp Rdx, int lane, const double* fc, const double* fl, const double* qc, const double* ql) {
  const bool pk = P.packed != 0;
  const int64_t* sj = s.sj;
  const int n = nr.n, j = nr.j;
  const double ut = un.t;
  const double dt = s.tf - s.to;
  const long long n3 = 3LL * n, n4 = 4LL * n;
  if (lane >= 1 && lane <= 11 && !(lane >= 5 && lane <= 7)) {
    double rh[3];
    for (int k = 0; k < 3; k++) rh[k] = fd_div_by(-(fl[k] - fc[k]), Rdx) * dt * ut / 2.0;
    const long long at = lane == 1 ? sj[GS_JV_MASS] : lane <= 4 ? sj[GS_JV_POS] + (lane - 2) * n3 : sj[GS_JV_QUAT] + (lane - 8) * n3;
    for (int k = 0; k < 3; k++) vals[at + 3LL * j + k] = rh[k];
  }
  if (lane == 12) {
    for (int k = 0; k < 3; k++) {
      const double rh_to = fc[k] * ut / 2.0;
      vals[sj[GS_JV_T] + 3LL * j + k] = rh_to;
      if (!pk) vals[sj[GS_JV_T] + n3 + 3LL * j + k] = -rh_to;
    }
  }
  if (lane == 14) {
    const GmRcp Rp = gm_rcp(un.pos);
    const double rh_vel = gm_div_by(-un.vel * dt * ut / 2.0, Rp);
    if (pk) {
      if (j == 0) vals[sj[GS_JP_VEL]] = rh_vel;
    } else {
      for (int k = 0; k < 3; k++) vals[sj[GS_JP_VEL] + 3LL * j + k] = rh_vel;
    }
    for (int k = 0; k < 3; k++) {
      const double rh_to = gm_div_by(s.vel[k] * un.vel * ut / 2.0, Rp);
      vals[sj[GS_JP_T] + 3LL * j + k] = rh_to;
      if (!pk) vals[sj[GS_JP_T] + n3 + 3LL * j + k] = -rh_to;
    }
  }
  if (!(nr.flags & GSF_HOLD)) {
    if (lane >= 1 && lane <= 6) {
      double rh[4];
      for (int a = 0; a < 4; a++) rh[a] = fd_div_by(-(ql[a] - qc[a]), Rdx) * dt * ut / 2.0;
      if (lane <= 4) {
        const int kk = lane - 1;
        const double d_diag = P.d_pool[nr.d_off + (long long)j * (n + 1) + (j + 1)];
        for (int a = 0; a < 4; a++) {
          const double base = (a == kk) ? d_diag : 0.0;
          const long long at = pk ? (4LL * j + a) * 4 + kk : (4LL * j + a) * (4LL * (n + 1)) + 4LL * (j + 1) + kk;
          vals[sj[GS_JQ_QUAT] + at] = base + rh[a];
        }
      } else {
        for (int a = 0; a < 4; a++) vals[sj[GS_JQ_U] + (lane - 5) * n4 + 4LL * j + a] = rh[a];
      }
    } else if (lane == 0) {
      for (int a = 0; a < 4; a++) {
        const double rh_to = qc[a] * ut / 2.0;
        vals[sj[GS_JQ_T] + 4LL * j + a] = rh_to;
        if (!pk) vals[sj[GS_JQ_T] + n4 + 4LL * j + a] = -rh_to;
      }
    }
  }
}
/* dx_dot<W> with the loads of four steps issued together, and optionally a one-column chain (the mass) in the same
 * loop: every chain still accumulates m ascending from 0.0 (DESIGN.md H2), so the bits are dx_dot's, but a part of the
 * vacuum kernel waits for loads (n + 1) / 4 times instead of (n + 1) / 2 times per array. */
template <int W, bool MASS>
P_HD void noair_dx_dot(const double* Drow, const double* xrows, const double* xmass, int n1, double* acc, double* acc_m) {
  double am = 0.0;
  for (int w = 0; w < W; w++) acc[w] = 0.0;
  int m = 0;
  for (; m + 4 <= n1; m += 4) {
    double d[4], xv[4][W], xm[4];
#pragma unroll
    for (int t = 0; t < 4; t++) {
      d[t] = Drow[m + t];
      for (int w = 0; w < W; w++) xv[t][w] = xrows[(long long)(m + t) * W + w];
      if (MASS) xm[t] = xmass[m + t];
    }
#pragma unroll
    for (int t = 0; t < 4; t++) {
      for (int w = 0; w < W; w++) acc[w] = gm_fma(d[t], xv[t][w], acc[w]);
      if (MASS) am = gm_fma(d[t], xm[t], am);
    }
  }
  for (; m < n1; m++) {
    const double d0 = Drow[m];
    for (int w = 0; w < W; w++) acc[w] = gm_fma(d0, xrows[(long long)m * W + w], acc[w]);
    if (MASS) am = gm_fma(d0, xmass[m], am);
  }
  if (MASS) *acc_m = am;
}
/* dyn_lh_item of the groups part 1 (velocity), 2 (position) or 3 (quaternion and mass) of a vacuum node computes */
P_HD void noair_lh(const PlanView& P, const double* x, const NodeRef& nr, int part, double* lh) {
  const int n1 = nr.n + 1, xa = nr.si[GS_XA], row = nr.row;
  const double* Drow = P.d_pool + nr.d_off + (long long)nr.j * n1;
  if (part == 1) {
    noair_dx_dot<3, false>(Drow, x + P.off_vel + 3 * xa, nullptr, n1, lh + 7, nullptr);
  } else if (part == 2) {
    noair_dx_dot<3, false>(Drow, x + P.off_pos + 3 * xa, nullptr, n1, lh, nullptr);
  } else {
    const bool qdot = !(nr.flags & GSF_HOLD), mdot = nr.flags & GSF_ENGINE_ON;
    if (qdot && mdot) {
      noair_dx_dot<4, true>(Drow, x + P.off_quat + 4 * xa, x + xa, n1, lh + 3, lh + 10);
      return;
    }
    if (qdot) noair_dx_dot<4, false>(Drow, x + P.off_quat + 4 * xa, nullptr, n1, lh + 3, nullptr);
    else
      for (int k = 0; k < 4; k++) lh[3 + k] = x[P.off_quat + 4 * row + k] - x[P.off_quat + 4 * xa + k];
    if (mdot) noair_dx_dot<1, false>(Drow, x + xa, nullptr, n1, lh + 10, nullptr);
    else lh[10] = x[row] - x[xa];
  }
}
/* phase B, warp `part` */
P_HD void dyn_noair_part(const PlanView& P, int scen, const double* x, double* vals, double* g, const NodeRef& nr, int part,
                         const NoairStage& s) {
  const Units un = scen_units(P, scen);
  const GmRcp Rv = gm_rcp(un.vel), Rdx = gm_rcp(un.dx);
  const bool hold = nr.flags & GSF_HOLD;
  double fc[3], fl[3], qc[4] = {0.0, 0.0, 0.0, 0.0}, ql[4] = {0.0, 0.0, 0.0, 0.0};
  /* centre column: pristine state, gravity at the pristine position */
  noair_col(s, 0, un, Rv, fc);
  if (!hold && part < 3) noair_quat_variant(s, 0, un, qc);
  if (part == 0) {
    dyn_noair_scatter(P, vals, nr, s, un, Rdx, 0, fc, fc, qc, qc);   /* eqcon_dyn_quat / t */
    dyn_noair_scatter(P, vals, nr, s, un, Rdx, 12, fc, fc, qc, qc);  /* eqcon_dyn_vel / t (analytic in vacuum) */
    dyn_noair_scatter(P, vals, nr, s, un, Rdx, 14, fc, fc, qc, qc);  /* eqcon_dyn_pos / velocity, t */
  }
  const int first = part == 0 ? 1 : part == 1 ? 3 : part == 2 ? 6 : 10;
  const int last = part == 0 ? 2 : part == 1 ? 5 : part == 2 ? 9 : 11;
  for (int lane = first; lane <= last; lane++) {
    if (lane == 7) continue;
    const bool vel_lane = lane >= 5 && lane <= 7;
    /* the position changes with lanes 2-4 and is fully restored from lane 5 on: lanes 8-11 share variant 4 */
    if (!vel_lane) noair_col(s, lane, un, Rv, fl);
    if (!hold && lane <= 6) noair_quat_variant(s, lane, un, ql);
    dyn_noair_scatter(P, vals, nr, s, un, Rdx, lane, fc, fl, qc, ql);
  }
  if (g && part > 0) { /* pair evaluation: the node's collocation defects, spread over the three lighter parts --
                          position | velocity | quaternion and mass (groups 0 | 2 | 1, 3 of dyn_lh_item) */
    double lh[11], qp[4] = {0.0, 0.0, 0.0, 0.0};
    if (part == 3 && !hold) noair_quat_variant(s, 7, un, qp);
    const int g0 = part == 2 ? 0 : part == 1 ? 2 : 1;
    noair_lh(P, x, nr, part, lh);
    dyn_res_finish(P, scen, x, g, nr, g0, lh, fc, qp);
    if (part == 3) dyn_res_finish(P, scen, x, g, nr, 3, lh, fc, qp);
  }
}
P_HD void dyn_noair_node(const PlanView& P, int scen, const double* x, double* vals, double* g, const NodeRef& nr) {
  NoairStage s;
  for (int part = 0; part < GV_PARTS; part++) dyn_noair_stage(P, scen, x, nr, part, s);
  for (int part = 0; part < GV_PARTS; part++) dyn_noair_part(P, scen, x, vals, g, nr, part, s);
}

/* ========================================================================= */
/* Jacobian kernel, DYN_GEN role (fallback): 16 lanes per node, every lane a  */
/* full right-hand side.  Used for sections whose reference_area is negative  */
/* (air formula, but no velocity / time finite differences: con_dynamics.py:  */
/* 257 vs :403,454).                                                          */
/* ========================================================================= */
GM_HD_INL void dyn_gen_phase(const PlanView& P, int scen, const double* x, double* vals, double* g, int start, int count,
                        int tid, int phase, const JacScratch& sm) {
  const int nl = tid >> 4, lane = tid & 15;
  if (nl >= count) return;
  const NodeRef nr = jac_node(P, start + nl);
  const Units un = scen_units(P, scen);
  const double dx = un.dx;
  const bool air = nr.flags & GSF_AIR, air_fd = nr.flags & GSF_AIR_FD, hold = nr.flags & GSF_HOLD;
  if (phase == 0) {
    const bool active = (lane <= 4) || (lane >= 8 && lane <= 11) || ((lane >= 5 && lane <= 7) && air_fd) ||
                        ((lane == 12 || lane == 13) && air_fd);
    if (active) {
      double v[11];
      dyn_col_state(P, x, nr.row, lane, air_fd, dx, v);
      const double to0 = x[P.off_t + nr.sec], tf0 = x[P.off_t + nr.sec + 1];
      const double to = (lane == 12) ? to0 + dx : to0;
      const double tf = (lane == 13) ? tf0 + dx : tf0;
      const SecParam sp = sec_param(P, scen, nr.sec);
      const Quat q = q4(v[7], v[8], v[9], v[10]);
      Vec3 f;
      if (air) {
        const double tn = time_node(P.tau_pool + nr.tau_off, nr.j + 1, to, tf);
        f = rhs_velocity_air(v[0], v3(v[1], v[2], v[3]), v3(v[4], v[5], v[6]), q, tn, sp, un, scen_tables(P, scen));
      } else {
        f = rhs_velocity_noair(v[0], v3(v[1], v[2], v[3]), q, sp, un);
      }
      double* o = sm.f + (nl * 14 + (lane < 14 ? lane : 0)) * 3;
      o[0] = f.x;
      o[1] = f.y;
      o[2] = f.z;
    }
    if (lane == 15 && !hold) dyn_quat_variants(P, x, nr, un, sm.q + nl * NQV * 4);
    if (lane == 14 && g)
      for (int grp = 0; grp < 4; grp++) dyn_lh_item(P, x, nr, grp, sm.lh + nl * 11);
  } else if (phase == 3) {
    const double* fc = sm.f + (nl * 14) * 3;
    const double* qc = sm.q + (nl * NQV) * 4;
    if (lane == 15) {
      if (g)
        for (int grp = 0; grp < 4; grp++) dyn_res_finish(P, scen, x, g, nr, grp, sm.lh + nl * 11, fc, qc + 7 * 4);
      return;
    }
    dyn_scatter(P, scen, x, vals, nr, lane, fc, fc + (lane < 14 ? lane : 0) * 3, qc, qc + (lane < 7 ? lane : 0) * 4);
  }
}

/* ========================================================================= */
/* Residual kernel, DYN role: GR_NODES consecutive nodes per block.           */
/*   phase 0: two threads per node: position part | rotation part             */
/*   phase 1: thread nl finishes the right-hand sides of its node             */
/*   phase 2: all threads sweep the (node, state column) items: D.X - rhs     */
/* reference: con_dynamics.py:34-63, 116-152, 216-289, 499-533                */
/* ========================================================================= */
/* phase 0: two threads per air node -- the position part and the rotation part of the
 * right-hand side do not depend on each other (the kernel is latency bound: one right-hand
 * side is a ~5 000-instruction dependent chain, splitting it halves the chain);
 * phase 1: one thread per node finishes its right-hand sides. */
P_HD void dyn_res_phase0(const PlanView& P, int scen, const double* x, int g0, int count, int tid, ResScratch& sm) {
  const int nl = tid >> 1, half = tid & 1;
  if (nl >= count) return;
  const NodeRef nr = res_node(P, g0 + nl);
  if (!(nr.flags & GSF_AIR)) return;
  const Units un = scen_units(P, scen);
  const int row = nr.row;
  const double px = x[P.off_pos + 3 * row] * un.pos, py = x[P.off_pos + 3 * row + 1] * un.pos,
               pz = x[P.off_pos + 3 * row + 2] * un.pos;
  if (half == 0) {
    const Tables tb = scen_tables(P, scen);
    pos_part(px, py, pz, tb.wind, tb.n_wind, PW_GRAVITY | PW_SOUND, sm.pp[nl]);
  } else {
    const double to = x[P.off_t + nr.sec], tf = x[P.off_t + nr.sec + 1];
    rotq_part(px, py, pz, time_node(P.tau_pool + nr.tau_off, nr.j + 1, to, tf), sm.rq[nl]);
  }
}

P_HD void dyn_res_phase1(const PlanView& P, int scen, const double* x, int g0, int count, int tid, ResScratch& sm) {
  if (tid >= count) return;
  const NodeRef nr = res_node(P, g0 + tid);
  const int row = nr.row;
  const Units un = scen_units(P, scen);
  const SecParam sp = sec_param(P, scen, nr.sec);
  const double m = x[row];
  const Vec3 p = v3(x[P.off_pos + 3 * row], x[P.off_pos + 3 * row + 1], x[P.off_pos + 3 * row + 2]);
  const Vec3 v = v3(x[P.off_vel + 3 * row], x[P.off_vel + 3 * row + 1], x[P.off_vel + 3 * row + 2]);
  const Quat q = q4(x[P.off_quat + 4 * row], x[P.off_quat + 4 * row + 1], x[P.off_quat + 4 * row + 2],
                    x[P.off_quat + 4 * row + 3]);
  Vec3 f;
  if (nr.flags & GSF_AIR) {
    double rp[RP_COLS];
    rot_wind(sm.rq[tid], sm.pp[tid][PP_WIND_N], sm.pp[tid][PP_WIND_E], rp);
    f = rhs_velocity_air_col(m, p, v, q, sm.pp[tid], rp, sp, un, scen_tables(P, scen));
  } else {
    f = rhs_velocity_noair(m, p, q, sp, un);
  }
  sm.f[tid][0] = f.x;
  sm.f[tid][1] = f.y;
  sm.f[tid][2] = f.z;
  if (!(nr.flags & GSF_HOLD)) {
    Quat d = rhs_quaternion(q, x[P.off_u + 2 * (nr.ua + nr.j)], x[P.off_u + 2 * (nr.ua + nr.j) + 1], un.u);
    sm.q[tid][0] = d.w;
    sm.q[tid][1] = d.x;
    sm.q[tid][2] = d.y;
    sm.q[tid][3] = d.z;
  }
}

/* D.X for one row of D and the W adjacent state columns of one state array (position 3, velocity 3,
 * quaternion 4, mass 1): acc[w] = fma(D[j][m], X[xa+m][w], acc[w]), m ascending.  The accumulation order
 * of each column is part of the numerical contract (DESIGN.md H2); the W chains are independent, so their
 * fixed latencies overlap, and one load of D[j][m] serves all of them. */
template <int W>
P_HD void dx_dot(const double* Drow, const double* xrows, int n1, double* acc) {
  for (int w = 0; w < W; w++) acc[w] = 0.0;
  int m = 0;
  for (; m + 2 <= n1; m += 2) { /* the loads of two steps are issued together */
    const double d0 = Drow[m], d1 = Drow[m + 1];
    double x0[W], x1[W];
    for (int w = 0; w < W; w++) x0[w] = xrows[(long long)m * W + w];
    for (int w = 0; w < W; w++) x1[w] = xrows[(long long)(m + 1) * W + w];
    for (int w = 0; w < W; w++) acc[w] = gm_fma(d0, x0[w], acc[w]);
    for (int w = 0; w < W; w++) acc[w] = gm_fma(d1, x1[w], acc[w]);
  }
  for (; m < n1; m++) {
    const double d0 = Drow[m];
    for (int w = 0; w < W; w++) acc[w] = gm_fma(d0, xrows[(long long)m * W + w], acc[w]);
  }
}

/* one column of a W-wide state array: the same chain as column k of dx_dot<W> */
P_HD double dx_dot_col(const double* Drow, const double* xcol, int stride, int n1) {
  double acc = 0.0;
  int m = 0;
  for (; m + 2 <= n1; m += 2) {
    const double d0 = Drow[m], d1 = Drow[m + 1];
    const double x0 = xcol[(long long)m * stride], x1 = xcol[(long long)(m + 1) * stride];
    acc = gm_fma(d0, x0, acc);
    acc = gm_fma(d1, x1, acc);
  }
  for (; m < n1; m++) acc = gm_fma(Drow[m], xcol[(long long)m * stride], acc);
  return acc;
}

/* The collocation defects of one (node, state array) item in two steps -- D.X (dyn_lh_item), then minus the
 * right-hand side (dyn_res_finish) -- so that the Jacobian kernel can compute the products while its long
 * phase-0 items run.  grp 0 position | 1 quaternion | 2 velocity | 3 mass; lh[11] = the node's products, laid
 * out position 3 | quaternion 4 | velocity 3 | mass 1; f3 / q4v: the node's velocity right-hand side and
 * quaternion kinematics at the pristine x.  Rows that are plain differences (engine off, held attitude) take
 * the difference as their "product".  Shared by the residual kernel (phase 2) and the pair evaluation. */
P_HD void dyn_lh_item(const PlanView& P, const double* x, const NodeRef& nr, int grp, double* lh) {
  const int n = nr.n, xa = nr.si[GS_XA], flags = nr.flags, j = nr.j, row = nr.row;
  const double* Drow = P.d_pool + nr.d_off + (long long)j * (n + 1);
  if (grp == 3) { /* mass: con_dynamics.py:53-61 */
    if (flags & GSF_ENGINE_ON) dx_dot<1>(Drow, x + xa, n + 1, lh + 10);
    else lh[10] = x[row] - x[xa];
  } else if (grp == 0) { /* position: :146 */
    dx_dot<3>(Drow, x + P.off_pos + 3 * xa, n + 1, lh);
  } else if (grp == 2) { /* velocity: :256 */
    dx_dot<3>(Drow, x + P.off_vel + 3 * xa, n + 1, lh + 7);
  } else if (flags & GSF_HOLD) { /* quaternion: :520-531 */
    for (int k = 0; k < 4; k++) lh[3 + k] = x[P.off_quat + 4 * row + k] - x[P.off_quat + 4 * xa + k];
  } else {
    dx_dot<4>(Drow, x + P.off_quat + 4 * xa, n + 1, lh + 3);
  }
}
/* column k of the velocity product alone (dyn_lh_item group 2) */
P_HD void dyn_lh_vel_col(const PlanView& P, const double* x, const NodeRef& nr, int k, double* lh) {
  const int n = nr.n, xa = nr.si[GS_XA];
  lh[7 + k] = dx_dot_col(P.d_pool + nr.d_off + (long long)nr.j * (n + 1), x + P.off_vel + 3 * xa + k, 3, n + 1);
}
P_HD void dyn_res_finish(const PlanView& P, int scen, const double* x, double* g, const NodeRef& nr, int grp,
                         const double* lh, const double* f3, const double* q4v) {
  const Units un = scen_units(P, scen);
  const double ut = un.t;
  const int32_t* si = nr.si;
  const int flags = nr.flags, j = nr.j, row = nr.row;
  const double to = x[P.off_t + nr.sec], tf = x[P.off_t + nr.sec + 1];
  const double dt = tf - to;
  if (grp == 3) {
    double r = lh[10];
    if (flags & GSF_ENGINE_ON) r = r - gm_div(-sec_param(P, scen, nr.sec).massflow, un.mass) * dt * ut / 2.0;
    g[si[GS_R_MASS] + j] = r;
  } else if (grp == 0) { /* :147-150 */
    const GmRcp Rp = gm_rcp(un.pos);
    for (int k = 0; k < 3; k++) {
      const double rh = gm_div_by(x[P.off_vel + 3 * row + k] * un.vel * dt * ut / 2.0, Rp);
      g[si[GS_R_POS] + 3 * j + k] = lh[k] - rh;
    }
  } else if (grp == 2) { /* :258-287 */
    for (int k = 0; k < 3; k++) {
      const double rh = f3[k] * dt * ut / 2.0;
      g[si[GS_R_VEL] + 3 * j + k] = lh[7 + k] - rh;
    }
  } else if (flags & GSF_HOLD) {
    for (int k = 0; k < 4; k++) g[si[GS_R_QUAT] + 4 * j + k] = lh[3 + k];
  } else { /* :525-530 */
    for (int k = 0; k < 4; k++) {
      const double rh = q4v[k] * dt * ut / 2.0;
      g[si[GS_R_QUAT] + 4 * j + k] = lh[3 + k] - rh;
    }
  }
}

/* phase 2 of the residual kernel.  One item per (node, state array), array-major (neighbouring threads run the
 * same array on neighbouring nodes), ordered position | quaternion | velocity | mass so that the two items a
 * thread takes (item, item + nthreads) carry 6 and 5 columns. */
P_HD void dyn_res_phase2(const PlanView& P, int scen, const double* x, double* g, int g0, int count, int tid,
                         int nthreads, const ResScratch& sm) {
  for (int item = tid; item < count * 4; item += nthreads) {
    const int grp = item / count, nl = item - grp * count;
    const NodeRef nr = res_node(P, g0 + nl);
    double lh[11];
    dyn_lh_item(P, x, nr, grp, lh);
    dyn_res_finish(P, scen, x, g, nr, grp, lh, sm.f[nl], sm.q[nl]);
  }
}

/* ========================================================================= */
/* Aero inequality jobs (con_aero.py:48-248, 311-756)                         */
/*   Jacobian lanes per constraint row:                                       */
/*   0 centre | 1-3 position | 4-6 velocity | 7-10 quaternion | 11 to | 12 tf */
/*   Same sharing as the dynamics: pv 0 base | 1-3 axis perturbed | 4 all     */
/*   restored; rv 0-4 nominal time | 5 to+dx | 6 tf+dx.                       */
/* ========================================================================= */
P_HD int aero_lane_pv(int lane) { return lane == 0 ? 0 : (lane <= 3 ? lane : 4); }
P_HD int aero_lane_rv(int lane) { return lane == 0 ? 0 : (lane <= 3 ? lane : (lane <= 10 ? 4 : lane - 6)); }

P_HD double aero_value(const PlanView& P, int scen, int kind, const double* v /*pos3 vel3 quat4*/, double t_e,
                       double limit) {
  const Units un = scen_units(P, scen);
  Vec3 pos = v3(v[0] * un.pos, v[1] * un.pos, v[2] * un.pos);
  Vec3 vel = v3(v[3] * un.vel, v[4] * un.vel, v[5] * un.vel);
  double t = t_e * un.t;
  return aero_quantity(kind, pos, vel, q4(v[6], v[7], v[8], v[9]), t, scen_tables(P, scen)) / limit;
}

P_HD void aero_load(const PlanView& P, const double* x, int row, double* v) {
  for (int k = 0; k < 3; k++) v[k] = x[P.off_pos + 3 * row + k];
  for (int k = 0; k < 3; k++) v[3 + k] = x[P.off_vel + 3 * row + k];
  for (int k = 0; k < 4; k++) v[6 + k] = x[P.off_quat + 4 * row + k];
}

/* state row + section times as the aero gradient finds them: residue left by the groups
 * that ran before it in `sens` (DESIGN.md H3) */
P_HD void aero_base(const PlanView& P, const double* x, int sec, int row, double* v, double* to, double* tf) {
  const double dx = P.un.dx;
  aero_load(P, x, row, v);
  *to = x[P.off_t + sec];
  *tf = x[P.off_t + sec + 1];
  if (P.rc_aero) {
    for (int k = 0; k < 3; k++) v[k] = residue_n(v[k], dx, P.rc_aero[P.off_pos + 3 * row + k]);
    for (int k = 0; k < 3; k++) v[3 + k] = residue_n(v[3 + k], dx, P.rc_aero[P.off_vel + 3 * row + k]);
    for (int k = 0; k < 4; k++) v[6 + k] = residue_n(v[6 + k], dx, P.rc_aero[P.off_quat + 4 * row + k]);
    *to = residue_n(*to, dx, P.rc_aero[P.off_t + sec]);
    *tf = residue_n(*tf, dx, P.rc_aero[P.off_t + sec + 1]);
  }
}

#ifndef GJA_SHARE_BASE
#define GJA_SHARE_BASE 1
#endif
GM_HD_INL void aero_phase(const PlanView& P, int scen, const double* x, double* vals, double* g, int start, int count, int tid,
                     int phase, const JacScratch& sm) {
  const Units un = scen_units(P, scen);
  const double dx = P.un.dx;
  /* pair evaluation (g != NULL): one more position / rotation variant and one more column per row, evaluated at
   * the PRISTINE state -- the value objfunc returns for the row (con_aero.py:89-248), out of the same launch */
  const int npv = g ? NPVA : NPV, nrv = g ? NRVA : NRV;
  if (phase == 0) {
    const bool is_a = tid < GJA_A_THREADS;
    const int per = is_a ? npv : nrv;
    const int step = is_a ? GJA_A_THREADS : GJ_THREADS - GJA_A_THREADS;
    for (int item = is_a ? tid : tid - GJA_A_THREADS; item < count * per; item += step) {
      const int nl = item / per, var = item - nl * per;
      const AeroRec ar = P.aero_rows[start + nl];
      double v[10], to, tf, p[3];
      const bool pristine = var == (is_a ? NPV : NRV);
      if (pristine) {
        aero_load(P, x, ar.row, v);
        to = x[P.off_t + ar.sec];
        tf = x[P.off_t + ar.sec + 1];
      } else {
        aero_base(P, x, ar.sec, ar.row, v, &to, &tf);
        /* the row's base state (what the gradient finds after the earlier groups' perturb / restore cycles) is the
         * same for all 13 columns of phase 2: kept in the quaternion scratch, which this role does not use */
        if (GJA_SHARE_BASE && is_a && var == 0)
          for (int k = 0; k < 10; k++) sm.q[nl * 10 + k] = v[k];
      }
      if (is_a) {
        pos_variant(v, pristine ? 0 : var, dx, p);
        const Tables tb = scen_tables(P, scen);
        pos_part(p[0] * un.pos, p[1] * un.pos, p[2] * un.pos, tb.wind, tb.n_wind, 0, sm.pp + (nl * NPVA + var) * PP_COLS);
      } else {
        pos_variant(v, pristine ? 0 : rv_pv(var), dx, p);
        if (var == 5) to = to + dx;
        if (var == 6) tf = tf + dx;
        const double tn = time_node(P.tau_pool + ar.tau_off, ar.r, to, tf);
        rotq_part(p[0] * un.pos, p[1] * un.pos, p[2] * un.pos, tn * un.t, sm.rq + (nl * NRVA + var) * RQ_COLS);
      }
    }
  } else if (phase == 2) {
    const int nlane = g ? 14 : 13;
    for (int item = tid; item < count * nlane; item += GJ_THREADS) {
      const int nl = item / nlane, lane = item - nl * nlane;
      const AeroRec ar = P.aero_rows[start + nl];
      const int kind = ar.kind, job = ar.job;
      const bool has_quat = kind != 1;
      if (!has_quat && lane >= 7 && lane <= 10) continue;
      double v[10];
      if (lane == 13) {
        aero_load(P, x, ar.row, v);
      } else if (GJA_SHARE_BASE) {
        for (int k = 0; k < 10; k++) v[k] = sm.q[nl * 10 + k]; /* aero_base of the row, from phase 0 */
      } else {
        double to, tf;
        aero_base(P, x, ar.sec, ar.row, v, &to, &tf);
      }
      if (lane != 0 && lane != 13) { /* the gradient works on a copy: columns leave residue inside the copy only */
        const int pidx = (lane <= 10) ? lane - 1 : 10;
        for (int w = 0; w < 10; w++) {
          if (!has_quat && w >= 6) continue;
          if (w < pidx) v[w] = residue(v[w], dx);
          else if (w == pidx) v[w] = v[w] + dx;
        }
      }
      double rp[RP_COLS];
      const double* pp = sm.pp + (nl * NPVA + (lane == 13 ? NPV : aero_lane_pv(lane))) * PP_COLS;
      rot_wind(sm.rq + (nl * NRVA + (lane == 13 ? NRV : aero_lane_rv(lane))) * RQ_COLS, pp[PP_WIND_N], pp[PP_WIND_E], rp);
      const Vec3 pos = v3(v[0] * un.pos, v[1] * un.pos, v[2] * un.pos);
      const Vec3 vel = v3(v[3] * un.vel, v[4] * un.vel, v[5] * un.vel);
      const double val = aero_quantity_col(kind, pos, vel, q4(v[6], v[7], v[8], v[9]),
                                           pp, rp) /
                         P.aero_f64[job * GA_F64_COLS + GA_LIMIT];
      sm.f[(nl * 14 + lane) * 3] = val;
    }
  } else {
    for (int item = tid; item < count * 12; item += GJ_THREADS) {
      const int lane = 1 + item / count, nl = item % count;
      const AeroRec ar = P.aero_rows[start + nl];
      const int64_t* aj = (P.packed ? P.aero_pk : P.aero_i64) + ar.job * GA_I64_COLS;
      const int kind = ar.kind, nk = ar.nk, r = ar.r;
      if (kind == 1 && lane >= 7 && lane <= 10) continue;
      const double gval = -fd_div(sm.f[(nl * 14 + lane) * 3] - sm.f[(nl * 14) * 3], dx); /* -dfdx (con_aero.py:439-461) */
      if (lane <= 3) vals[aj[GA_J_POS] + (long long)(lane - 1) * nk + r] = gval;
      else if (lane <= 6) vals[aj[GA_J_VEL] + (long long)(lane - 4) * nk + r] = gval;
      else if (lane <= 10) vals[aj[GA_J_QUAT] + (long long)(lane - 7) * nk + r] = gval;
      else if (lane == 11) vals[aj[GA_J_T] + r] = gval;
      else vals[aj[GA_J_T] + nk + r] = gval;
    }
    if (g)
      for (int nl = GJ_THREADS - 1 - tid; nl < count; nl += GJ_THREADS) { /* 1 - f: con_aero.py:89-248 */
        const AeroRec ar = P.aero_rows[start + nl];
        g[ar.row0 + ar.r] = 1.0 - sm.f[(nl * 14 + 13) * 3];
      }
  }
}

/* residual kernel: one thread per aero row, pristine inputs: 1 - f (con_aero.py:89-248) */
P_HD void aero_res(const PlanView& P, int scen, const double* x, double* g, const AeroRec& ar) {
  double v[10];
  aero_load(P, x, ar.row, v);
  const double tn = time_node(P.tau_pool + ar.tau_off, ar.r, x[P.off_t + ar.sec], x[P.off_t + ar.sec + 1]);
  g[ar.row0 + ar.r] = 1.0 - aero_value(P, scen, ar.kind, v, tn, P.aero_f64[ar.job * GA_F64_COLS + GA_LIMIT]);
}

/* ========================================================================= */
/* Event-point jobs: waypoint LLH / IIP / antenna rows, terminal orbit,       */
/* perigee user constraint.  16 lanes per job in the Jacobian kernel.         */
/* ========================================================================= */
struct EvtOut {
  double v[3];
};

/* evaluate the leaf of an event job: pe/ve non-dimensional state row, t_e non-dimensional */
P_HD EvtOut evt_leaf(const PlanView& P, int scen, int type, const double* ef, const double* pe, const double* ve,
                     double t_e, int ei_comp = 0, int nrow = 1) {
  const Units un = scen_units(P, scen);
  EvtOut o;
  o.v[0] = o.v[1] = o.v[2] = 0.0;
  Vec3 pos = v3(pe[0] * un.pos, pe[1] * un.pos, pe[2] * un.pos);
  Vec3 vel = v3(ve[0] * un.vel, ve[1] * un.vel, ve[2] * un.vel);
  if (type == GE_LLH) { /* con_waypoint.py:565-566 */
    Vec3 llh = eci2geodetic_deg(pos, t_e * un.t);
    o.v[0] = llh.x; o.v[1] = llh.y; o.v[2] = llh.z;
  } else if (type == GE_IIP) { /* :214-218 */
    Vec3 llh = iip_from_eci_deg(pos, vel, t_e * un.t);
    o.v[0] = llh.x; o.v[1] = llh.y; o.v[2] = llh.z;
  } else if (type == GE_ANT) { /* :45-51 */
    o.v[0] = sin_elevation(pos, t_e * un.t, v3(ef[GE_A0], ef[GE_A1], ef[GE_A2]));
  } else if (type == GE_TERM) { /* con_init_terminal_knot.py:362-370 */
    o.v[0] = (orbit_energy(pos, vel) / ef[GE_A0]) - 1.0;
    o.v[1] = (angular_momentum(pos, vel) / ef[GE_A1]) - 1.0;
    o.v[2] = inclination_rad(pos, vel) - ef[GE_A2];
  } else { /* GE_USER_ORBIT: rows q / scale - offset (example/user_constraints.py:133-137 is perigee / 6378137 - 1) */
    const int codes = ei_comp;
    for (int r = 0; r < nrow && r < 3; r++)
      o.v[r] = (orbit_quantity((codes >> (8 * r)) & 0xff, pos, vel) / ef[GE_A0 + 2 * r]) - ef[GE_A0 + 2 * r + 1];
  }
  return o;
}

P_HD double evt_form_value(int form, double v, double ref, double den) {
  switch (form) {
    case GEF_DIFF_OVER_DEN: return (v - ref) / den;
    case GEF_NEG_DIFF_OVER_DEN: return -(v - ref) / den;
    case GEF_RATIO_M1: return (v / ref) - 1.0;
    case GEF_NEG_RATIO_P1: return -(v / ref) + 1.0;
    case GEF_REF_MINUS_OVER_DEN: return (ref - v) / den;
    default: return v - ref;
  }
}
P_HD double evt_form_grad(int form, double gfd, double ref, double den) {
  switch (form) {
    case GEF_DIFF_OVER_DEN: return gfd / den;
    case GEF_NEG_DIFF_OVER_DEN: return -gfd / den;
    case GEF_RATIO_M1: return gfd / ref;
    case GEF_NEG_RATIO_P1: return -gfd / ref;
    case GEF_REF_MINUS_OVER_DEN: return -gfd / den;
    default: return gfd;
  }
}

/* residual kernel: one thread per event job, pristine inputs */
P_HD void evt_res(const PlanView& P, int scen, const double* x, double* g, int job) {
  const int32_t* ei = P.evt_i32 + job * GE_I32_COLS;
  const double* ef = P.evt_f64 + job * GE_F64_COLS;
  const int type = ei[GE_TYPE], srow = ei[GE_SROW];
  const double t_e = (ei[GE_TIDX] >= 0) ? x[P.off_t + ei[GE_TIDX]] : 0.0;
  EvtOut o = evt_leaf(P, scen, type, ef, x + P.off_pos + 3 * srow, x + P.off_vel + 3 * srow, t_e, ei[GE_COMP], ei[GE_NROW]);
  if (type == GE_TERM) {
    for (int r = 0; r < ei[GE_NROW]; r++) g[ei[GE_ROW] + r] = o.v[r];
  } else if (type >= GE_USER_ORBIT) {
    for (int r = 0; r < ei[GE_NROW]; r++) g[ei[GE_ROW] + r] = o.v[r];
  } else {
    g[ei[GE_ROW]] = evt_form_value(ei[GE_FORM], o.v[ei[GE_COMP]], ef[GE_REF], ef[GE_DEN]);
  }
}

/* Jacobian kernel lane maps (perturbation order of the reference):
 *   LLH / ANT : 0 centre | 1-3 pos j | 4 t                       (con_waypoint.py:54-66, 570-578)
 *   IIP       : 0 centre | 1 p0 2 v0 3 p1 4 v1 5 p2 6 v2 | 7 t   (:225-236, interleaved)
 *   TERM      : 0 centre | 1-3 pos j | 4-6 vel j                  (con_init_terminal_knot.py:391-399)
 *   USER_ORBIT: 0 base | 1-6 FD of p0 p1 p2 v0 v1 v2 | 7-12 background after k restores
 *               (jac_fd.py:54-60 restricted to the six variables the function reads).  Lane 7 holds k = 0, the
 *               base state again: (g_base - g_base) / dx is what jac_fd gives every variable visited before the
 *               first one the function reads -- +0, or NaN where g_base is not finite.  k = 1 is never needed
 *               (the three position components are visited back to back), so the slot is free for it. */
P_HD int evt_n_lanes(int type) {
  return type == GE_IIP ? 8 : (type == GE_TERM ? 7 : (type == GE_USER_ORBIT ? 13 : 5));
}

P_HD void evt_jac_phase1(const PlanView& P, int scen, const double* x, int job, int tid, bool pair, const JacScratch& sm) {
  const int lane = tid & 15;
  const int32_t* ei = P.evt_i32 + job * GE_I32_COLS;
  const double* ef = P.evt_f64 + job * GE_F64_COLS;
  const int type = ei[GE_TYPE], srow = ei[GE_SROW];
  if (lane == 15) { /* pair evaluation: the leaf at the PRISTINE state -- objfunc's row (evt_res) */
    if (!pair) return;
    const double t0 = (ei[GE_TIDX] >= 0) ? x[P.off_t + ei[GE_TIDX]] : 0.0;
    EvtOut o = evt_leaf(P, scen, type, ef, x + P.off_pos + 3 * srow, x + P.off_vel + 3 * srow, t0, ei[GE_COMP], ei[GE_NROW]);
    sm.f[3 * tid + 0] = o.v[0];
    sm.f[3 * tid + 1] = o.v[1];
    sm.f[3 * tid + 2] = o.v[2];
    return;
  }
  if (lane >= evt_n_lanes(type)) return;
  const double dx = P.un.dx;
  double s[6]; /* pos[3], vel[3] base state = r^rc(x) */
  for (int k = 0; k < 3; k++) s[k] = residue_n(x[P.off_pos + 3 * srow + k], dx, ei[GE_RC0 + k]);
  for (int k = 0; k < 3; k++) s[3 + k] = residue_n(x[P.off_vel + 3 * srow + k], dx, ei[GE_RC0 + 3 + k]);
  double t_e = (ei[GE_TIDX] >= 0) ? residue_n(x[P.off_t + ei[GE_TIDX]], dx, ei[GE_RC0 + 6]) : 0.0;
  /* order[] = sequence in which the reference perturbs the six state variables */
  int order[6], nvar;
  if (type == GE_IIP) {
    order[0] = 0; order[1] = 3; order[2] = 1; order[3] = 4; order[4] = 2; order[5] = 5;
    nvar = 6;
  } else if (type == GE_TERM || type == GE_USER_ORBIT) {
    for (int k = 0; k < 6; k++) order[k] = k;
    nvar = 6;
  } else {
    for (int k = 0; k < 3; k++) order[k] = k;
    nvar = 3;
  }
  if (lane >= 1) {
    int n_restored, perturbed = -1;
    if (lane <= nvar) { /* FD lane for variable order[lane-1] */
      n_restored = lane - 1;
      perturbed = order[lane - 1];
    } else if (type == GE_USER_ORBIT) { /* background lanes 7..12: k = lane-6 restores done, except k = 0 on lane 7 */
      n_restored = lane == 7 ? 0 : lane - 6;
    } else { /* the t lane: every variable already restored */
      n_restored = nvar;
      t_e = t_e + dx;
    }
    for (int k = 0; k < n_restored; k++) s[order[k]] = residue(s[order[k]], dx);
    if (perturbed >= 0) s[perturbed] = s[perturbed] + dx;
  }
  EvtOut o = evt_leaf(P, scen, type, ef, s, s + 3, t_e, ei[GE_COMP], ei[GE_NROW]);
  sm.f[3 * tid + 0] = o.v[0];
  sm.f[3 * tid + 1] = o.v[1];
  sm.f[3 * tid + 2] = o.v[2];
}

P_HD void evt_jac_phase2(const PlanView& P, double* vals, double* g, int job, int tid, const JacScratch& sm) {
  const int lane = tid & 15;
  const int32_t* ei = P.evt_i32 + job * GE_I32_COLS;
  const int64_t* ej = (P.packed ? P.evt_pk : P.evt_i64) + job * GE_I64_COLS;
  const double* ef = P.evt_f64 + job * GE_F64_COLS;
  const int type = ei[GE_TYPE];
  if (lane == 15) { /* objfunc's row(s) of this job, as evt_res writes them */
    if (!g) return;
    const double* o = sm.f + 3 * tid;
    if (type == GE_TERM) {
      for (int r = 0; r < ei[GE_NROW]; r++) g[ei[GE_ROW] + r] = o[r];
    } else if (type >= GE_USER_ORBIT) {
      for (int r = 0; r < ei[GE_NROW]; r++) g[ei[GE_ROW] + r] = o[r];
    } else {
      g[ei[GE_ROW]] = evt_form_value(ei[GE_FORM], o[ei[GE_COMP]], ef[GE_REF], ef[GE_DEN]);
    }
    return;
  }
  if (lane == 0 || lane >= evt_n_lanes(type)) return;
  const double dx = P.un.dx;
  const int c = tid & ~15;
  if (type == GE_TERM) { /* (f_p - f_c)/dx, COO order: column-major over the nRow rows */
    const int nrow = ei[GE_NROW];
    const int64_t base = (lane <= 3) ? ej[GE_J_POS] + (long long)(lane - 1) * nrow
                                     : ej[GE_J_VEL] + (long long)(lane - 4) * nrow;
    for (int r = 0; r < nrow; r++) vals[base + r] = fd_div(sm.f[3 * tid + r] - sm.f[3 * c + r], dx);
    return;
  }
  if (type == GE_USER_ORBIT) { /* aux tail, per row: fd[6] then background[6] */
    for (int r = 0; r < ei[GE_NROW]; r++)
      vals[ej[GE_J_POS] + r * GE_USER_AUX + (lane - 1)] = fd_div(sm.f[3 * tid + r] - sm.f[3 * c + r], dx);
    return;
  }
  const int comp = ei[GE_COMP], form = ei[GE_FORM];
  const double gfd = fd_div(sm.f[3 * tid + comp] - sm.f[3 * c + comp], dx);
  const double val = evt_form_grad(form, gfd, ef[GE_REF], ef[GE_DEN]);
  if (type == GE_IIP) {
    if (lane == 7) vals[ej[GE_J_T]] = val;
    else if (lane & 1) vals[ej[GE_J_POS] + (lane - 1) / 2] = val;
    else vals[ej[GE_J_VEL] + (lane - 2) / 2] = val;
  } else {
    if (lane == 4) vals[ej[GE_J_T]] = val;
    else vals[ej[GE_J_POS] + (lane - 1)] = val;
  }
}

/* ========================================================================= */
/* Linear rows (init / time / knot / rate / stage mass / kick / time order)   */
/* ========================================================================= */
P_HD void lin_res(const PlanView& P, int scen, const double* x, double* g, int k) {
  const int32_t* li = P.lin_i32 + k * GL_I32_COLS;
  const double* lf = P.lin_f64 + k * GL_F64_COLS;
  const double a = (li[GL_IDX_PLUS] >= 0) ? x[li[GL_IDX_PLUS]] * lf[GL_SCALE_PLUS] : 0.0;
  const double b = (li[GL_IDX_MINUS] >= 0) ? x[li[GL_IDX_MINUS]] * lf[GL_SCALE_MINUS] : 0.0;
  const double c = P.lin_const_scen ? P.lin_const_scen[(long long)scen * P.n_lin + k] : lf[GL_CONST];
  /* signed zeros as the reference's expressions give them: -u (the kick rows) and u_j - u_k are not 0 - u and
   * (u_j - u_k) + 0, which turn -0 into +0 */
  const double d = (li[GL_IDX_PLUS] >= 0) ? a - b : -b;
  g[li[GL_ROW]] = (c != 0.0) ? d + c : d;
}

/* ========================================================================= */
/* Block dispatch.  Jacobian blocks run GJ_PHASES phases with a block barrier  */
/* between them; residual blocks run three (only the dynamics role uses 0, 2).  */
/* ROLES is the mask of roles an instantiation of the Jacobian kernel contains  */
/* (the shipped kernel: all of them; subsets exist for measurements).  The      */
/* dispatch and the role functions are forced inline: the kernel calls them     */
/* once per phase with a constant phase number, and a copy left as a real call  */
/* takes the phase at run time and the plan view / scratch through local memory */
/* (measured: 0.29 -> 0.42 ms, 600 MB of local-memory traffic per launch).      */
/* ========================================================================= */
#define JR_HEAVY ((1 << BR_DYN_AIR) | (1 << BR_AERO))
#define JR_LIGHT ((1 << BR_DYN_NOAIR) | (1 << BR_DYN_GEN) | (1 << BR_EVT) | (1 << BR_LIN))
#define JR_ALL (JR_HEAVY | JR_LIGHT)
P_HD void lin_res(const PlanView& P, int scen, const double* x, double* g, int k);
template <int ROLES>
GM_HD_INL void jac_block_phase(const PlanView& P, int scen, const int32_t* bt, const double* x, double* vals, double* g,
                          int tid, int phase, const JacScratch& sm) {
  const int start = bt[BT_START], count = bt[BT_COUNT], role = bt[BT_ROLE];
  if ((ROLES >> BR_DYN_AIR & 1) && role == BR_DYN_AIR) dyn_air_phase(P, scen, x, vals, g, start, count, tid, phase, sm);
  if ((ROLES >> BR_AERO & 1) && role == BR_AERO) aero_phase(P, scen, x, vals, g, start, count, tid, phase, sm);
  if ((ROLES >> BR_DYN_NOAIR & 1) && role == BR_DYN_NOAIR) dyn_noair_phase(P, scen, x, vals, g, start, count, tid, phase, sm);
  if ((ROLES >> BR_DYN_GEN & 1) && role == BR_DYN_GEN) dyn_gen_phase(P, scen, x, vals, g, start, count, tid, phase, sm);
  if ((ROLES >> BR_EVT & 1) && role == BR_EVT && (tid >> (GJ_EVT_PER_WARP ? 5 : 4)) < count &&
      (!GJ_EVT_PER_WARP || (tid & 31) < 16)) {
    const int job = tid >> (GJ_EVT_PER_WARP ? 5 : 4);
    const int slot = job * 16 + (tid & (GJ_EVT_PER_WARP ? 31 : 15)); /* the 16-lane numbering the job functions use */
    if (phase == 0) evt_jac_phase1(P, scen, x, start + job, slot, g != nullptr, sm);
    else if (phase == 3) evt_jac_phase2(P, vals, g, start + job, slot, sm);
  }
  /* pair evaluation only: the linear rows and the objective (the launch leaves these blocks out otherwise) */
  if ((ROLES >> BR_LIN & 1) && role == BR_LIN && phase == 3 && g) {
    if (tid < count) lin_res(P, scen, x, g, start + tid);
    if (start == 0 && tid == 0) g[0] = P.payload_mode ? -x[0] : x[P.off_t + P.S]; /* cost_gradient.py:29-34 */
  }
}
/* roles whose phase 2 is empty (the kernel skips that barrier); phase 1 is empty for every role */
P_HD bool jac_role_two_phase(int role) { return role == BR_EVT || role == BR_DYN_GEN || role == BR_LIN; }

P_HD void res_block_phase0(const PlanView& P, int scen, const int32_t* bt, const double* x, int tid, ResScratch& sm) {
  if (bt[BT_ROLE] == BR_DYN) dyn_res_phase0(P, scen, x, bt[BT_START], bt[BT_COUNT], tid, sm);
}
P_HD void res_block_phase1(const PlanView& P, int scen, const int32_t* bt, const double* x, double* g, int tid,
                           ResScratch& sm) {
  switch (bt[BT_ROLE]) {
    case BR_DYN: dyn_res_phase1(P, scen, x, bt[BT_START], bt[BT_COUNT], tid, sm); break;
    case BR_AERO:
      if (tid < bt[BT_COUNT]) {
        aero_res(P, scen, x, g, P.aero_rows[bt[BT_START] + tid]);
      }
      break;
    case BR_EVT:
      if (tid < bt[BT_COUNT]) evt_res(P, scen, x, g, bt[BT_START] + tid);
      break;
    case BR_LIN:
      if (tid < bt[BT_COUNT]) lin_res(P, scen, x, g, bt[BT_START] + tid);
      if (bt[BT_START] == 0 && tid == 0) /* objective: cost_gradient.py:29-34 */
        g[0] = P.payload_mode ? -x[0] : x[P.off_t + P.S];
      break;
    default: break;
  }
}
P_HD void res_block_phase2(const PlanView& P, int scen, const int32_t* bt, const double* x, double* g, int tid,
                           int nthreads, const ResScratch& sm) {
  if (bt[BT_ROLE] == BR_DYN) dyn_res_phase2(P, scen, x, g, bt[BT_START], bt[BT_COUNT], tid, nthreads, sm);
}

#endif /* GELATO_B200_JOBS_H_ */
