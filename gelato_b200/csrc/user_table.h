/* user_table.h -- the result-table user constraints (include/gelato_b200.h: GT_*, gelato_b200.plan.TableAtEvent):
 * any of the 34 per-node quantities of output.h, at the first node of a named event, with jac_fd's dense Jacobian.
 *
 * One job = GT_LANES evaluations of output_row, one per lane of a warp (k_user_table) or one after the other (the host
 * emulator, tests/emu):
 *   lane 0        the base state r^rc(x)
 *   lanes 1-12    jac_fd's column of read variable lane - 1 (xdict order: mass, position 3, velocity 3, quaternion 4, t):
 *                 the read variables before it restored once more, itself perturbed by +dx
 *   lanes 13-17   the background states: k = 1, 4, 7, 11, 12 of the read variables restored, nothing perturbed
 *   lane 18       the pristine state (objfunc's rows; pair and residual evaluations)
 * Each lane evaluates the whole row of 34 columns once; every constraint row of the job picks its column from it, and
 * the quotients against lane 0 go to the row's GT_AUX slots.  These functions stay out of the block kernels
 * (jobs.h): output_row (Vincenty loop, IIP iteration, Euler angles) would enter the 448-thread kernel that every
 * pair step runs. */
#ifndef GELATO_B200_USER_TABLE_H_
#define GELATO_B200_USER_TABLE_H_

#include "jobs.h"
#include "output.h"

static_assert(GO_COLS == GT_COLUMNS, "column codes are output_row's outputs");

#define GT_NREAD 12    /* variables the function reads */
#define GT_PRISTINE 18 /* the lane of objfunc's rows */
#define GT_LANES 19

/* the table jobs on the device (or the host): the GelatoPlanDesc tables, and each row's offset in the packed output */
struct TabView {
  int n_tab;
  const int32_t* i32;
  const double* f64;
  const int32_t* col;
  const int64_t* aux;
  const double* sf;
  const int64_t* pk;
};

/* restores done on background lane 13 + b: after the event's mass, position, velocity, quaternion and t */
P_HD int table_bg_restores(int b) { return b == 0 ? 1 : (b == 1 ? 4 : (b == 2 ? 7 : (b == 3 ? 11 : 12))); }

/* the 34 columns of lane `lane` of job `job`, scenario `scen` (parameter blocks), decision vector x */
P_HD void table_lane_eval(const PlanView& P, const TabView& T, int scen, const double* x, int job, int lane, double* out) {
  const int32_t* ti = T.i32 + (long long)job * GT_I32_COLS;
  const int srow = ti[GT_SROW], i = ti[GT_TIDX];
  double s[GT_NREAD];
  s[0] = x[srow];
  for (int k = 0; k < 3; k++) s[1 + k] = x[P.off_pos + 3 * srow + k];
  for (int k = 0; k < 3; k++) s[4 + k] = x[P.off_vel + 3 * srow + k];
  for (int k = 0; k < 4; k++) s[7 + k] = x[P.off_quat + 4 * srow + k];
  s[11] = x[P.off_t + i];
  if (lane != GT_PRISTINE) {
    const double dx = P.un.dx;
    for (int k = 0; k < GT_NREAD; k++) s[k] = residue_n(s[k], dx, ti[GT_RC0 + k]);
    const int n_restored = lane <= GT_NREAD ? (lane > 0 ? lane - 1 : 0) : table_bg_restores(lane - GT_NREAD - 1);
    for (int k = 0; k < n_restored; k++) s[k] = residue(s[k], dx);
    if (lane >= 1 && lane <= GT_NREAD) s[lane - 1] = s[lane - 1] + dx;
  }
  const Units un = scen_units(P, scen);
  const SecParam sp = sec_param(P, scen, i);
  const double* tf = T.f64 + (long long)job * GT_F64_COLS;
  output_row(s[0] * un.mass, v3(s[1] * un.pos, s[2] * un.pos, s[3] * un.pos), v3(s[4] * un.vel, s[5] * un.vel, s[6] * un.vel),
             q4(s[7], s[8], s[9], s[10]), s[11] * un.t, sp.thrust, sp.ref_area, sp.nozzle_area, scen_tables(P, scen),
             tf[GT_LAT0], tf[GT_LON0], out);
}

/* row r of job `job` from its lane's columns: column / scale - offset (the reference's expression) */
P_HD double table_row_value(const TabView& T, int job, int r, const double* out) {
  const int row = T.i32[(long long)job * GT_I32_COLS + GT_R0] + r;
  return out[T.col[row]] / T.sf[GT_SF_COLS * row + GT_SCALE] - T.sf[GT_SF_COLS * row + GT_OFFSET];
}

/* what lane `lane` writes for row r, given its value v and lane 0's v0: the pristine lane objfunc's row into g, the
 * others their quotient into the row's aux slots of vals (COO or packed layout, P.packed) */
P_HD void table_lane_store(const PlanView& P, const TabView& T, int job, int r, int lane, double v, double v0, double* vals,
                           double* g) {
  const int32_t* ti = T.i32 + (long long)job * GT_I32_COLS;
  if (lane == GT_PRISTINE) {
    g[ti[GT_ROW] + r] = v;
    return;
  }
  const int row = ti[GT_R0] + r;
  vals[(P.packed ? T.pk[row] : T.aux[row]) + (lane == 0 ? GT_AUX - 1 : lane - 1)] = fd_div(v - v0, P.un.dx);
}

#endif /* GELATO_B200_USER_TABLE_H_ */
