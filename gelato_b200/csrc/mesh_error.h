/* mesh_error.h -- the integral-form collocation error estimate of each section (Patterson, Hager & Rao 2015; DESIGN.md
 * section 11), as per-thread functions.
 *
 * Section i has n LGR nodes over the support points s = {-1, tau_1 .. tau_n}.  Its test grid has M points tau'_l with
 * four host-built tables (include/gelato_b200.h: GelatoMeshGridDesc): tau_t[M], the Lagrange basis P[M][n+1] over s
 * (states), the basis Q[M][n] over tau_1 .. tau_n (controls) and the integration matrix I[M][M] of the test grid.  Per
 * test point l the state X_l and controls U_l are interpolated and rh_l, the right-hand-side term of dyn_res_finish,
 * is evaluated there (mesh_point).  Per state component c the estimate is then
 *     err = max_l |X_0 + sum_k I[l][k] rh_k - X_l| / (1 + max_l |X_l|)
 * with X_0 the section's first state row (mesh_component).  Every sum is a fused multiply-add chain with ascending
 * index from 0.0, and max and division are exact, so the result has one value: the kernels, the host emulator
 * (tests/emu/emu.cpp) and the oracle (tests/mesh_oracle.py) agree bit for bit.
 *
 * The path check runs on the same grid: the aero constraints' residual 1 - f at every test point of every aero job over
 * a whole section (mesh_path_point), and its minimum per job (mesh_path_min).  Min and 1 - f are exact, so it too has
 * one value.
 *
 * The path rows put those residuals into the NLP as inequality rows, on a grid of their own (gelato_plan_set_path_rows),
 * with their Jacobian by the chain rule through the interpolation: the derivative along each state component of the
 * interpolated state (a finite-difference quotient, path_lane_quot) times the P entry of each state row.
 */
#ifndef GELATO_B200_MESH_ERROR_H_
#define GELATO_B200_MESH_ERROR_H_

#include "jobs.h"

#define MESH_STATE 11            /* mass | position 3 | velocity 3 | quaternion 4 */
#define MESH_PT (2 * MESH_STATE) /* doubles per test point in the scratch: X_l, then rh_l */

/* one section of a test grid: M test points, the first one's index in the plan's list of test points, and the offset
 * of the section's tables in the pool */
struct MeshSec {
  int32_t m, pt0;
  int64_t off;
};
/* one test point: its section and its index inside the section */
struct MeshPt {
  int32_t sec, l;
};
/* one test point of the path check: an aero job over a whole section and the index of the test point in that section */
struct PathPt {
  int32_t job, l;
};

struct MeshTabs {
  const double *tau, *P, *Q, *I;
};
/* the pool is laid out tau_t[M] | P[M][n+1] | Q[M][n] | I[M][M] from the section's offset */
P_HD MeshTabs mesh_tabs(const double* pool, const MeshSec& ms, int n) {
  MeshTabs t;
  t.tau = pool + ms.off;
  t.P = t.tau + ms.m;
  t.Q = t.P + (long long)ms.m * (n + 1);
  t.I = t.Q + (long long)ms.m * n;
  return t;
}

/* component c of state row `row` */
P_HD double mesh_state(const PlanView& P, const double* x, int row, int c) {
  if (c == 0) return x[row];
  if (c < 4) return x[P.off_pos + 3 * row + c - 1];
  if (c < 7) return x[P.off_vel + 3 * row + c - 4];
  return x[P.off_quat + 4 * row + c - 7];
}

/* Test point l of section `sec`: xl[11] = the interpolated state, rh[11] = the right-hand-side term of each state
 * component there, with the operations of dyn_res_finish (engine-off mass and held attitude: 0). */
P_HD void mesh_point(const PlanView& P, int scen, const double* x, int sec, const MeshTabs& tb, int l, double* xl,
                     double* rh) {
  const int32_t* si = P.sec_i32 + sec * GS_I32_COLS;
  const int n = si[GS_N], ua = si[GS_UA], xa = si[GS_XA], flags = si[GS_FLAGS];
  const double* Prow = tb.P + (long long)l * (n + 1);
  const double* Qrow = tb.Q + (long long)l * n;
  dx_dot<1>(Prow, x + xa, n + 1, xl);
  dx_dot<3>(Prow, x + P.off_pos + 3 * xa, n + 1, xl + 1);
  dx_dot<3>(Prow, x + P.off_vel + 3 * xa, n + 1, xl + 4);
  dx_dot<4>(Prow, x + P.off_quat + 4 * xa, n + 1, xl + 7);
  double ul[2];
  dx_dot<2>(Qrow, x + P.off_u + 2 * ua, n, ul);

  const Units un = scen_units(P, scen);
  const SecParam sp = sec_param(P, scen, sec);
  const double ut = un.t;
  const double to = x[P.off_t + sec], tf = x[P.off_t + sec + 1];
  const double dt = tf - to;
  rh[0] = (flags & GSF_ENGINE_ON) ? gm_div(-sp.massflow, un.mass) * dt * ut / 2.0 : 0.0;
  const GmRcp Rp = gm_rcp(un.pos);
  for (int k = 0; k < 3; k++) rh[1 + k] = gm_div_by(xl[4 + k] * un.vel * dt * ut / 2.0, Rp);
  const Vec3 p = v3(xl[1], xl[2], xl[3]), v = v3(xl[4], xl[5], xl[6]);
  const Quat q = q4(xl[7], xl[8], xl[9], xl[10]);
  Vec3 f;
  if (flags & GSF_AIR) f = rhs_velocity_air(xl[0], p, v, q, time_node(tb.tau, l + 1, to, tf), sp, un, scen_tables(P, scen));
  else f = rhs_velocity_noair(xl[0], p, q, sp, un);
  rh[4] = f.x * dt * ut / 2.0;
  rh[5] = f.y * dt * ut / 2.0;
  rh[6] = f.z * dt * ut / 2.0;
  if (flags & GSF_HOLD) {
    for (int k = 0; k < 4; k++) rh[7 + k] = 0.0;
  } else {
    const Quat d = rhs_quaternion(q, ul[0], ul[1], un.u);
    rh[7] = d.w * dt * ut / 2.0;
    rh[8] = d.x * dt * ut / 2.0;
    rh[9] = d.y * dt * ut / 2.0;
    rh[10] = d.z * dt * ut / 2.0;
  }
}

/* v[10] = position | velocity | quaternion of section `sec` interpolated at test point l with the chains of mesh_point
 * (its xl[1..10]) */
P_HD void mesh_path_state(const PlanView& P, const double* x, int sec, const MeshTabs& tb, int l, double* v) {
  const int32_t* si = P.sec_i32 + sec * GS_I32_COLS;
  const int n = si[GS_N], xa = si[GS_XA];
  const double* Prow = tb.P + (long long)l * (n + 1);
  dx_dot<3>(Prow, x + P.off_pos + 3 * xa, n + 1, v);
  dx_dot<3>(Prow, x + P.off_vel + 3 * xa, n + 1, v + 3);
  dx_dot<4>(Prow, x + P.off_quat + 4 * xa, n + 1, v + 6);
}

/* ========================================================================= */
/* Path rows (DESIGN.md section 11): the aero constraints as NLP rows at the  */
/* test points of a grid of their own.  Per row 16 lanes:                     */
/*   0 centre | 1-10 state component (position 3 | velocity 3 | quaternion 4)*/
/*   | 11 to | 12 tf | 13-15 idle                                             */
/* ========================================================================= */
#define PATH_LANES 16
enum { PR_POS = 0, PR_VEL, PR_QUAT, PR_T, PR_OFFS };
/* one path row: aero job, test point of the job's section, and where each variable's entries start in the row values
 * of one scenario (PR_QUAT: -1 for max-q, which has none); plan_host.h: build_path_rows */
struct PathRow {
  int32_t job, l;
  int64_t off[PR_OFFS];
};

/* f / L of lane `lane` of a path row at step dx, v = mesh_path_state of the row's test point: lane 0 f(v, tn) (dx
 * unused), lanes 1-10 f(v + dx e_(lane-1), tn), 11 and 12 f(v, tn) with to + dx and tf + dx.  The centre is the path
 * check's f at that test point. */
P_HD double path_lane_f(const PlanView& P, int scen, const double* x, int job, const MeshTabs& tb, int l, const double* v,
                        int lane, double dx) {
  const int32_t* ai = P.aero_i32 + job * GA_I32_COLS;
  const int sec = ai[GA_SECTION];
  double w[10];
#pragma unroll
  for (int k = 0; k < 10; k++) w[k] = k == lane - 1 ? v[k] + dx : v[k]; /* no dynamic index: w stays in registers */
  double to = x[P.off_t + sec], tf = x[P.off_t + sec + 1];
  if (lane == 11) to = to + dx;
  else if (lane == 12) tf = tf + dx;
  return aero_value(P, scen, ai[GA_KIND], w, time_node(tb.tau, l + 1, to, tf), P.aero_f64[job * GA_F64_COLS + GA_LIMIT]);
}

/* The path check (DESIGN.md section 11): one test point of an aero job.  The job's section is interpolated at test
 * point l (mesh_path_state), and the residual is the expression aero_res gives objfunc's row at a node: pristine x,
 * the time of the test point, the scenario's units and wind table (path_lane_f's centre lane).  At a test point that is
 * a node it is that row's value, bit for bit. */
P_HD double mesh_path_point(const PlanView& P, int scen, const double* x, int job, const MeshTabs& tb, int l) {
  double v[10];
  mesh_path_state(P, x, P.aero_i32[job * GA_I32_COLS + GA_SECTION], tb, l, v);
  return 1.0 - path_lane_f(P, scen, x, job, tb, l, v, 0, 0.0);
}

/* the derivative of the row 1 - f / L along lane `lane` (1-12), f0 = the centre: -fd_div(f(step) - f0, step); central
 * differences (DESIGN.md H6) average that quotient at +step and at -step */
P_HD double path_lane_quot(const PlanView& P, int scen, const double* x, int job, const MeshTabs& tb, int l, const double* v,
                           int lane, double f0, int central, double step) {
  /* one evaluation site for both steps: the device build of two inlined copies of the evaluation returned wrong -step
   * quotients for the state lanes (the t lanes and forward mode were right) */
  double q = 0.0;
#pragma unroll 1
  for (int s = 0; s <= central; s++) {
    const double h = s ? -step : step;
    const double qs = -fd_div(path_lane_f(P, scen, x, job, tb, l, v, lane, h) - f0, h);
    q = s ? fd_central(q, qs) : qs;
  }
  return q;
}

/* the entries of lane `lane` (1-12) of path row `pr` into one scenario's row values: a state lane writes P[l][m] * q for
 * the section's state rows m = 0..n at (m, component), lanes 11 / 12 write q itself */
P_HD void path_lane_store(const PathRow& pr, const double* Prow, int n, int lane, double q, double* vals) {
  if (lane >= 11) {
    vals[pr.off[PR_T] + (lane - 11)] = q;
    return;
  }
  const int var = lane <= 3 ? PR_POS : (lane <= 6 ? PR_VEL : PR_QUAT);
  const int w = var == PR_QUAT ? 4 : 3, c = lane <= 3 ? lane - 1 : (lane <= 6 ? lane - 4 : lane - 7);
  double* out = vals + pr.off[var] + c;
  for (int m = 0; m <= n; m++) out[(long long)w * m] = Prow[m] * q;
}

/* min and argmin of r[0 .. m) as numpy.min / numpy.argmin give them: ties go to the first, a NaN wins (the first NaN);
 * m == 0 (an "initial" job, a point constraint with nothing between nodes): +inf at -1 */
P_HD void mesh_path_min(const double* r, int m, double* res, int32_t* at) {
  double best = gm_inf();
  int32_t k_best = -1;
  for (int k = 0; k < m; k++) {
    const double v = r[k];
    if (k == 0 || v < best || (v != v && best == best)) {
      best = v;
      k_best = k;
    }
  }
  *res = best;
  *at = k_best;
}

/* max as numpy's: a NaN operand makes the result NaN */
P_HD double mesh_max(double a, double b) { return (b > a || b != b) ? b : a; }

/* The estimate of state component c of section `sec`: pts = the section's M test points as mesh_point left them,
 * MESH_PT doubles each. */
P_HD double mesh_component(const PlanView& P, const double* x, int sec, const MeshTabs& tb, int M, const double* pts, int c) {
  const double x0 = mesh_state(P, x, P.sec_i32[sec * GS_I32_COLS + GS_XA], c);
  double emax = 0.0, xmax = 0.0;
  for (int l = 0; l < M; l++) {
    const double* Irow = tb.I + (long long)l * M;
    double acc = 0.0;
    for (int k = 0; k < M; k++) acc = gm_fma(Irow[k], pts[(long long)k * MESH_PT + MESH_STATE + c], acc);
    const double xl = pts[(long long)l * MESH_PT + c];
    emax = mesh_max(emax, gm_fabs((x0 + acc) - xl));
    xmax = mesh_max(xmax, gm_fabs(xl));
  }
  return gm_div(emax, 1.0 + xmax);
}

#endif /* GELATO_B200_MESH_ERROR_H_ */
