/* gelato_b200.h -- C ABI of the B200 NLP-callback engine.
 *
 * This is the boundary that replaces the reference's five pybind11 extension
 * modules (/root/reference/src/pybind_dynamics.cpp:108-114, pybind_utils.cpp:28-48,
 * pybind_coordinate.cpp:28-78, pybind_IIP.cpp:53-57,
 * pybind_USStandardAtmosphere.cpp:28-35) AND the Python loops around them
 * (/root/reference/lib/con_*.py): instead of ~230 by-value leaf calls per
 * Jacobian, the host describes the whole transcribed problem once (a "plan") and
 * then makes ONE call (one kernel launch) per `objfunc` (/root/reference/Trajectory_Optimization.py:194-242)
 * and ONE per `sens` (:245-312) -- or one for both (gelato_eval_pair_*).
 *
 * Plain pointers and sizes only; no torch / numpy / Eigen types.  All functions
 * return 0 on success and a negative code on failure (gelato_last_error() gives
 * the text).  There is no CPU fallback: without a CUDA device every evaluation
 * entry point fails with GELATO_ERR_CUDA.
 *
 * Decision vector x (length n_vars), reference order
 * (/root/reference/Trajectory_Optimization.py:318-352):
 *     mass[M] | position[3M] | velocity[3M] | quaternion[4M] | u[2N] | t[S+1]
 * Residual vector g (length n_rows): g[0] = objective, then the constraint
 * groups in the order the plan's row offsets define (the reference's funcs order).
 * Jacobian value vector vals (length n_vals): the reference's COO `data` arrays
 * concatenated group by group, variable by variable, followed by a small
 * auxiliary tail (user-constraint finite differences).
 */
#ifndef GELATO_B200_H_
#define GELATO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GELATO_OK 0
#define GELATO_ERR_ARG (-1)
#define GELATO_ERR_CUDA (-2)
#define GELATO_ERR_ALLOC (-3)

/* ---- section table columns (one row per collocation section) ------------- */
enum {
  GS_N = 0,    /* LGR nodes in the section */
  GS_UA,       /* first control row (reference PSparams.get_index: ua) */
  GS_XA,       /* first state row (xa); rows xa .. xa+n */
  GS_FLAGS,    /* GSF_* */
  GS_D_OFF,    /* offset (doubles) of D[n][n+1] in the D pool */
  GS_TAU_OFF,  /* offset of tau[n] in the tau pool */
  GS_R_MASS,   /* first residual row of eqcon_dyn_mass for this section */
  GS_R_POS,
  GS_R_VEL,
  GS_R_QUAT,
  GS_I32_COLS
};
enum {
  GSF_ENGINE_ON = 1, /* params[i]["engineOn"] (con_dynamics.py:53) */
  GSF_AIR = 2,       /* reference_area != 0.0 (con_dynamics.py:257) */
  GSF_AIR_FD = 4,    /* reference_area > 0.0  (con_dynamics.py:403,454) */
  GSF_HOLD = 8       /* attitude in {hold, vertical} (con_dynamics.py:520) */
};
/* offsets into vals of the x-dependent Jacobian blocks of a section (-1: absent) */
enum {
  GS_JP_VEL = 0, /* eqcon_dyn_pos / velocity : 3n           (con_dynamics.py:180-183) */
  GS_JP_T,       /* eqcon_dyn_pos / t        : 3n to + 3n tf (:186-195) */
  GS_JV_MASS,    /* eqcon_dyn_vel / mass     : 3n           (:372-380) */
  GS_JV_POS,     /* eqcon_dyn_vel / position : 3 x 3n       (:383-400) */
  GS_JV_VEL,     /* eqcon_dyn_vel / velocity : 9 x n(n+1)   (:418-428) */
  GS_JV_QUAT,    /* eqcon_dyn_vel / quaternion: 4 x 3n      (:431-449) */
  GS_JV_T,       /* eqcon_dyn_vel / t        : 3n to + 3n tf (:482-489) */
  GS_JQ_QUAT,    /* eqcon_dyn_quat / quaternion: 4n x 4(n+1) (:591-597) */
  GS_JQ_U,       /* eqcon_dyn_quat / u       : 2 x 4n       (:600-613) */
  GS_JQ_T,       /* eqcon_dyn_quat / t       : 4n to + 4n tf (:616-625) */
  GS_I64_COLS
};
enum { GS_THRUST = 0, GS_MASSFLOW, GS_REF_AREA, GS_NOZZLE_AREA, GS_F64_COLS };

/* ---- linear rows: g[row] = (sp*x[ip] - sm*x[im]) + c  (index -1 = absent) -- */
enum { GL_ROW = 0, GL_IDX_PLUS, GL_IDX_MINUS, GL_I32_COLS };
enum { GL_SCALE_PLUS = 0, GL_SCALE_MINUS, GL_CONST, GL_F64_COLS };

/* ---- aero inequality jobs (con_aero.py) ----------------------------------- */
enum { GA_KIND = 0 /* 0 alpha, 1 q, 2 q-alpha */, GA_SECTION, GA_NK, GA_ROW0, GA_I32_COLS };
enum { GA_J_POS = 0, GA_J_VEL, GA_J_QUAT, GA_J_T, GA_I64_COLS };
enum { GA_LIMIT = 0, GA_F64_COLS };

/* ---- event-point jobs (con_waypoint.py, con_init_terminal_knot.py:329-405,
 *      user constraint built-ins) ------------------------------------------- */
enum { GE_LLH = 0, GE_IIP = 1, GE_ANT = 2, GE_TERM = 3, GE_USER_ORBIT = 4, GE_N_TYPES };
#define GE_USER_PERIGEE GE_USER_ORBIT /* round-1 name: the one-row perigee-radius case */
/* GE_USER_ORBIT: a built-in user constraint (/root/reference/lib/con_user.py:33-42 + jac_fd.py:29-62) on orbit
 * quantities of the state at the first node of a named event, up to three rows: row r = q / scale - offset with the
 * quantity code in byte r of GE_COMP (GEQ_*) and scale / offset in GE_A0 + 2r, GE_A0 + 2r + 1.  It leaves GE_USER_AUX
 * values per row in the auxiliary tail of vals: 6 finite-difference quotients (position, velocity) and the 6
 * "background" quotients jac_fd's perturb / restore protocol gives every variable the function does not read
 * (after 0, 2, 3, 4, 5, 6 of the read variables are restored; the first is +0, or NaN where the row is not finite). */
#define GE_USER_AUX 12
enum {
  GEQ_PERIGEE_RADIUS = 0, /* a (1 - e)       Coordinate.cpp:197-245 orbital_elements */
  GEQ_APOGEE_RADIUS,      /* a (1 + e) */
  GEQ_SEMI_MAJOR_AXIS,    /* a */
  GEQ_ECCENTRICITY,       /* e */
  GEQ_INCLINATION_DEG,    /* acos of the orbit normal's z, in degrees (wrapper_coordinate.hpp:204) */
  GEQ_ORBIT_ENERGY,       /* v^2 / 2 - mu / r    wrapper_coordinate.hpp:224-250 */
  GEQ_ANGULAR_MOMENTUM,   /* |r x v| */
  GEQ_N
};
enum {
  GE_TYPE = 0,
  GE_TIDX,    /* index into t (section number), -1 if unused */
  GE_SROW,    /* state row (position/velocity row index) */
  GE_COMP,    /* component of the leaf's output used by this row */
  GE_FORM,    /* GEF_* value formula */
  GE_ROW,     /* residual row (first row for GE_TERM) */
  GE_NROW,    /* rows produced (GE_TERM: 2 or 3; others 1) */
  GE_RC0,     /* 7 residue counts: pos[3], vel[3], t  (see DESIGN.md "H3") */
  GE_I32_COLS = GE_RC0 + 7
};
enum {
  GEF_DIFF_OVER_DEN = 0, /*  (v - ref)/den                */
  GEF_NEG_DIFF_OVER_DEN, /* -(v - ref)/den                */
  GEF_RATIO_M1,          /*  v/ref - 1                    */
  GEF_NEG_RATIO_P1,      /* -(v/ref) + 1                  */
  GEF_REF_MINUS_OVER_DEN,/*  (ref - v)/den                */
  GEF_MINUS_REF          /*  v - ref                      */
};
enum { GE_J_POS = 0, GE_J_VEL, GE_J_T, GE_I64_COLS };
enum { GE_REF = 0, GE_DEN, GE_A0, GE_A1, GE_A2, GE_A3, GE_A4, GE_A5, GE_F64_COLS };

/* ---- result-table user constraints (gelato_b200.plan.TableAtEvent) -------------------------------------------
 * A built-in user constraint on columns of the reference's result table (the 34 outputs of gelato_leaf_output_table)
 * at the first node of event i (state row srow = index_start_u(i) + i, time t[i] * unit_t, section i's thrust /
 * reference_area / nozzle_area, the scenario's wind table, the plan's CA table, the launch site's lat / lon):
 *     g[row + r] = column_r / scale_r - offset_r.
 * The reference applies jac_fd (jac_fd.py:29-62) to it.  The function reads 12 variables, in xdict order: mass[srow],
 * position[3 srow + 0..2], velocity[3 srow + 0..2], quaternion[4 srow + 0..3], t[i].  Each of its rows leaves GT_AUX
 * values in vals, at its own offset:
 *     0..11   the finite-difference quotient of each read variable (the variables visited before it restored, itself
 *             perturbed by +dx)
 *     12..16  the "background" quotients jac_fd gives the variables the function does not read: k = 1, 4, 7, 11, 12 of
 *             the read variables restored, nothing perturbed
 *     17      k = 0: (base - base) / dx, +0 or NaN where the base value is not finite
 * all from the base state r^rc(x) (the 12 residue counts GT_RC0.. of the groups evaluated earlier).  One kernel of its
 * own (k_user_table: a warp per scenario and job) evaluates them next to the Jacobian kernel. */
#define GT_AUX 18
#define GT_COLUMNS 34 /* column codes: the order of gelato_leaf_output_table's outputs */
enum {
  GT_SROW = 0, /* state row of the event's first node */
  GT_TIDX,     /* event index i: t[i], section i's parameters; 0 <= i < S */
  GT_ROW,      /* first residual row */
  GT_NROW,     /* rows of the job (>= 1) */
  GT_R0,       /* its first row in the row tables tab_col / tab_aux / tab_sf */
  GT_RC0,      /* 12 residue counts: mass, position[3], velocity[3], quaternion[4], t */
  GT_I32_COLS = GT_RC0 + 12
};
enum { GT_LAT0 = 0, GT_LON0, GT_F64_COLS }; /* LaunchCondition lat / lon (deg), for downrange */
enum { GT_SCALE = 0, GT_OFFSET, GT_SF_COLS };

typedef struct GelatoPlanDesc {
  /* sizes */
  int32_t n_sections, n_nodes; /* S, N;  M = N + S */
  int32_t n_rows;              /* length of g (objective included) */
  int64_t n_vals;              /* length of vals (aux tail included) */
  int32_t payload_mode;        /* 1: objective = -mass[0]; 0: objective = t[S] */
  /* sections */
  const int32_t* sec_i32; /* [S][GS_I32_COLS] */
  const int64_t* sec_i64; /* [S][GS_I64_COLS] */
  const double* sec_f64;  /* [S][GS_F64_COLS] */
  const double* d_pool;   /* concatenated row-major D blocks */
  int64_t d_pool_len;
  const double* tau_pool;
  int64_t tau_pool_len;
  /* tables */
  const double* wind; /* [n_wind][3] altitude, wind_n, wind_e */
  int32_t n_wind;
  const double* ca; /* [n_ca][2] mach, CA */
  int32_t n_ca;
  /* units (/root/reference/Trajectory_Optimization.py:153-167) */
  double unit_mass, unit_pos, unit_vel, unit_u, unit_t, dx;
  /* linear rows */
  int32_t n_lin;
  const int32_t* lin_i32;
  const double* lin_f64;
  /* aero jobs */
  int32_t n_aero;
  const int32_t* aero_i32;
  const int64_t* aero_i64;
  const double* aero_f64;
  const uint8_t* rc_aero; /* [n_vars] residue counts seen by the aero groups (may be NULL) */
  /* event jobs */
  int32_t n_evt;
  const int32_t* evt_i32;
  const int64_t* evt_i64;
  const double* evt_f64;
  /* Jacobian template: constants and D entries, length n_vals */
  const double* vals_template;
  /* sorted positions in vals of the x-dependent slots (what the Jacobian kernel rewrites on
   * every call); may be NULL, then the update-mode entry points are unavailable */
  const int64_t* xdep_idx;
  int64_t n_xdep;
  /* result-table user constraints (GT_* above); n_tab = 0 / NULL tables: none */
  int32_t n_tab;
  const int32_t* tab_i32; /* [n_tab][GT_I32_COLS] */
  const double* tab_f64;  /* [n_tab][GT_F64_COLS] */
  int32_t n_tab_rows;
  const int32_t* tab_col; /* [n_tab_rows] column code, 0 <= code < GT_COLUMNS */
  const int64_t* tab_aux; /* [n_tab_rows] first of the row's GT_AUX slots in vals */
  const double* tab_sf;   /* [n_tab_rows][GT_SF_COLS] */
} GelatoPlanDesc;

/* per-scenario overrides for batched evaluation (NULL members = shared) */
typedef struct GelatoScenarioDesc {
  int32_t n_scen;
  const double* sec_f64;       /* [n_scen][S][GS_F64_COLS] */
  const double* wind;          /* [n_scen][n_wind][3] */
  const double* unit_mass;     /* [n_scen] */
  const double* lin_const;     /* [n_scen][n_lin] */
  const double* vals_template; /* [n_scen][n_vals] */
} GelatoScenarioDesc;

typedef struct GelatoPlan GelatoPlan;

const char* gelato_last_error(void);
int gelato_device_count(void);

int gelato_plan_create(const GelatoPlanDesc* desc, int device, GelatoPlan** out);
int gelato_plan_set_scenarios(GelatoPlan* plan, const GelatoScenarioDesc* sc);
int gelato_plan_destroy(GelatoPlan* plan);
int32_t gelato_plan_n_vars(const GelatoPlan* plan);
int32_t gelato_plan_n_rows(const GelatoPlan* plan);
int64_t gelato_plan_n_vals(const GelatoPlan* plan);
/* thread blocks per scenario: which = 0 residual kernel | 1 Jacobian kernel | 2 / 3 its heavy / light roles' blocks
 * | 4 Jacobian kernel of a pair evaluation (+ the linear-row blocks) */
int32_t gelato_plan_n_blocks(const GelatoPlan* plan, int which);
/* kernels launched by this plan so far (bench.py's gpu_launches) */
int64_t gelato_plan_launch_count(const GelatoPlan* plan);

/* How the Jacobian's finite-difference values are formed (DESIGN.md H3, H6).
 *   GELATO_FD_FORWARD (default)  the reference's forward differences with the plan's dx, bit for bit;
 *   GELATO_FD_CENTRAL            central differences with step h: every finite-difference value is
 *                                (q(+h) + q(-h)) * 0.5, q(+-h) being the forward protocol run with step +-h.
 *                                Analytic and constant slots, sparsity, COO order and the packed layout do not
 *                                change; objfunc values do not depend on the mode.  It costs a second Jacobian
 *                                launch and one averaging pass (DESIGN.md H6 gives the measured cost), plus
 *                                n_scen x n_pack doubles of plan-owned device scratch.
 * gelato_plan_set_fd: mode and step (`step` is ignored for FORWARD, which always uses the plan's dx); a bad mode, or a
 * central step that is not finite and in (0, 1e-3], returns GELATO_ERR_ARG and leaves the plan unchanged.  Every entry
 * point that returns Jacobian values honours the mode (host, update, packed, _ids and _dev calls), except
 * gelato_eval_pair_packed_range_dev, which refuses central mode, and the measurement helpers gelato_time_kernel and
 * gelato_launch_kernel_dev, which always launch the forward kernels once.  Central _dev calls use the plan's scratch:
 * calls on one plan must not overlap on different streams.
 * gelato_plan_get_fd: the current mode and step (FORWARD: the plan's dx). */
enum { GELATO_FD_FORWARD = 0, GELATO_FD_CENTRAL = 1 };
int gelato_plan_set_fd(GelatoPlan* plan, int32_t mode, double step);
int gelato_plan_get_fd(const GelatoPlan* plan, int32_t* mode, double* step);

/* Host-buffer entry points (what the drop-in objfunc / sens call): copy x to the
 * device, run ONE fused kernel, copy the result back.  n_scen = 1 for a single NLP;
 * x is [n_scen][n_vars], g [n_scen][n_rows], vals [n_scen][n_vals].  Buffers obtained
 * from gelato_host_alloc (page-locked) are DMA'd directly; any other host memory is
 * staged through the plan's own page-locked buffers. */
int gelato_eval_residuals(GelatoPlan* plan, const double* x, double* g, int32_t n_scen);
int gelato_eval_jacobian(GelatoPlan* plan, const double* x, double* vals, int32_t n_scen);

/* Subset batches: batch slot k is evaluated with the parameter blocks of configured scenario
 * scen_ids[k] (0 <= scen_ids[k] < n_scen of gelato_plan_set_scenarios; repeats allowed).  This is what a
 * coalescing server needs: of many concurrent solves, those that happen to be waiting for a callback are
 * evaluated together in one launch (gelato_b200/server.py). */
int gelato_eval_residuals_ids(GelatoPlan* plan, const double* x, double* g, int32_t n_scen, const int32_t* scen_ids);
int gelato_eval_jacobian_ids(GelatoPlan* plan, const double* x, double* vals, int32_t n_scen, const int32_t* scen_ids);

/* Update mode for drivers that keep one host Jacobian buffer per scenario batch alive across
 * calls (a batched solve): most of vals never changes (D entries, +-1, unit constants -- 87 % of
 * the slots at 1 000 nodes), so only the x-dependent slots cross PCIe.
 *   gelato_jacobian_template     fills vals[n_scen][n_vals] with the constant slots (once per buffer);
 *   gelato_eval_jacobian_update  runs the Jacobian kernel and moves only the x-dependent slots into
 *                                vals (page-locked vals: long runs copied into place, scattered slots
 *                                packed and scattered by a pool of host threads or written from the
 *                                device; pageable vals: all packed, copied and scattered by the pool);
 *                                every other slot of vals is left as it was.
 * After the two calls vals holds exactly what gelato_eval_jacobian returns. */
/* gelato_eval_pair_update: `objfunc` and `sens` of the same decision vectors in one call -- x is uploaded
 * once, one pair evaluation (see gelato_eval_pair_dev), g is copied back whole and vals is updated as by
 * gelato_eval_jacobian_update.  Results are those of the two separate calls. */
int64_t gelato_plan_n_xdep(const GelatoPlan* plan);
int gelato_jacobian_template(GelatoPlan* plan, double* vals, int32_t n_scen);
int gelato_eval_jacobian_update(GelatoPlan* plan, const double* x, double* vals, int32_t n_scen);
int gelato_eval_pair_update(GelatoPlan* plan, const double* x, double* g, double* vals, int32_t n_scen);
/* Scattered x-dependent slots of a page-locked `vals` (gelato_host_alloc).  on == 0 (default on hosts with 8 or
 * more hardware threads): packed on the device, copied as one block, scattered by the host thread pool.
 * on != 0 (default on smaller hosts): written straight into `vals` from the device (zero-copy over PCIe, no
 * host thread touches the buffer; isolated 8-byte writes reach ~6 GB/s).  Pageable buffers always take the
 * packed route. */
int gelato_set_update_zero_copy(GelatoPlan* plan, int32_t on);
/* Update mode is pipelined over `n` slices of the batch (slice k's upload and kernels overlap slice k-1's
 * device->host traffic and host scatter); 0 = chosen from the batch size (one slice per 16 scenarios, at most 8). */
int gelato_set_update_slices(GelatoPlan* plan, int32_t n);
/* Measurement only: device times (ms) of the transfer pieces of update mode, each alone (out_ms[6]: long-run 2-D
 * copies, zero-copy kernel, both, pack + contiguous copy of the scattered slots, one contiguous copy of all
 * x-dependent bytes, the residual copy).  `vals` page-locked, after a gelato_eval_*_update call. */
int gelato_probe_update(GelatoPlan* plan, double* vals, int32_t n_scen, int reps, float* out_ms);
/* host threads used by the scatter of update mode (default: min(16, hardware threads)) */
int gelato_set_host_threads(GelatoPlan* plan, int32_t n_threads);

/* Packed mode: what a batched driver that assembles its own sparse matrices should call (the consumer gathers,
 * nobody scatters).  The Jacobian kernels write only the INDEPENDENT x-dependent values of each scenario,
 * contiguously (n_pack per scenario: the node-diagonal entries of the dense D (x) I blocks as dense arrays, one
 * value instead of 3n for eqcon_dyn_pos/velocity, no `tf` halves that are exact negations of the `to` halves --
 * about 15 % fewer values than the x-dependent COO slots), and g and packed come back as contiguous copies.
 *   gelato_plan_n_pack        n_pack
 *   gelato_plan_packed_map    for each of the n_xdep x-dependent COO slots, ascending (full_slot == xdep_idx): the
 *                             packed value it holds and its sign: vals[full_slot[i]] = sgn[i] * packed[src[i]]
 *                             (sgn = +-1.0; with the constant slots of gelato_jacobian_template this reproduces
 *                             gelato_eval_jacobian bit for bit -- a CSR / KKT assembly composes this map with its
 *                             own once and then gathers straight from `packed`)
 *   gelato_eval_pair_packed   objfunc + sens of the same x: g[n_scen][n_rows] and packed[n_scen][n_pack]
 *   gelato_eval_jacobian_packed  sens only
 *   gelato_eval_pair_packed_ids  subset batches (see gelato_eval_residuals_ids)
 * Host buffers; page-locked ones (gelato_host_alloc) are DMA'd directly; pipelined over slices of the batch. */
int64_t gelato_plan_n_pack(const GelatoPlan* plan);
int gelato_plan_packed_map(const GelatoPlan* plan, int64_t* full_slot, int64_t* src, double* sgn);
int gelato_eval_pair_packed(GelatoPlan* plan, const double* x, double* g, double* packed, int32_t n_scen);
int gelato_eval_jacobian_packed(GelatoPlan* plan, const double* x, double* packed, int32_t n_scen);
int gelato_eval_pair_packed_ids(GelatoPlan* plan, const double* x, double* g, double* packed, int32_t n_scen,
                                const int32_t* scen_ids);

/* Mesh error estimate (DESIGN.md section 11): how well the dynamics hold BETWEEN the collocation nodes.  For each section
 * the state and controls are interpolated at M test points tau'_l, the right-hand side of the collocation defects is
 * evaluated there, integrated with the test grid's integration matrix from the section's first state row, and compared
 * with the interpolated state:
 *     err[s][i][c] = max_l |X_0,c + sum_k I[l][k] rh_k,c - X_l,c| / (1 + max_l |X_l,c|)
 * for scenario s, section i and state component c (mass | position 3 | velocity 3 | quaternion 4).  Engine-off mass
 * and held attitude have no right-hand side: their estimate is the spread of the interpolated state around X_0.
 * gelato_plan_set_mesh_grid: the test grid, copied to the device.  m[i] (>= 1) test points of section i, whose tables
 * lie in `pool` from offset off[i] on, laid out
 *     tau_t[M] | P[M][n+1] | Q[M][n] | I[M][M]
 * (n = the section's LGR nodes): the test points in [-1, 1], the Lagrange basis over {-1, tau_1 .. tau_n} (states) and
 * over tau_1 .. tau_n (controls) at the test points, and the inverse of the test grid's LGR differentiation matrix
 * without its first column (gelato_b200/mesh.py: grid_tables builds them with M = n + 1).  M < 1, a table outside the
 * pool or a value in the pool that is not finite returns GELATO_ERR_ARG and leaves the plan unchanged.
 * gelato_eval_mesh_error: host buffers, x [n_scen][n_vars], err [n_scen][S][11] (page-locked buffers are DMA'd
 * directly, others staged).  _dev: device pointers, enqueued on `stream` (NULL = the plan's own), not synchronised.
 * Both use the scenario blocks of gelato_plan_set_scenarios, refuse an n_scen beyond them as every entry point does, and
 * refuse calls before a grid is set.  Two launches per call (DESIGN.md section 11 gives the measured cost); the _dev call
 * uses plan-owned scratch (n_scen x sum(M) x 22 doubles): calls on one plan must not overlap on different streams.
 * Intervals (a section made of several LGR intervals, h-refinement; optional, trailing): n_int[i] (>= 1) intervals of
 * section i; per interval, in section order, int_m its test points (they partition the section's M, in order) and
 * int_base the support column (0..n) it integrates from: strictly increasing in a section, 0 for its first interval.
 * Interval k of a section has the estimate of the formula above over its own test points l, with X_0 the state row
 * xa + int_base[k] and the sum over its own k only (its block of I; P and Q rows may be interval-local bases).  The
 * section's err is the max over its intervals.  n_int == NULL: one interval per section from column 0, the estimate
 * above.  n_int < 1, interval test points that do not add up to m, or a base out of range, not increasing or not 0 for
 * a section's first interval returns GELATO_ERR_ARG and leaves the plan unchanged.
 * gelato_eval_mesh_error_intervals: err_int [n_scen][sum n_int][11], each interval's estimate, with the buffers,
 * scenario blocks, scratch and refusals of gelato_eval_mesh_error; _dev as gelato_eval_mesh_error_dev. */
typedef struct GelatoMeshGridDesc {
  const int32_t* m;   /* [S] test points of each section */
  const int64_t* off; /* [S] offset (doubles) of each section's tables in pool */
  const double* pool;
  int64_t pool_len;
  const int32_t* n_int;    /* [S] intervals of each section, or NULL: one each */
  const int32_t* int_m;    /* [sum n_int] test points of each interval */
  const int32_t* int_base; /* [sum n_int] support column each interval integrates from */
} GelatoMeshGridDesc;
int gelato_plan_set_mesh_grid(GelatoPlan* plan, const GelatoMeshGridDesc* grid);
int gelato_eval_mesh_error(GelatoPlan* plan, const double* x, double* err, int32_t n_scen);
int gelato_eval_mesh_error_dev(GelatoPlan* plan, const double* x_dev, double* err_dev, int32_t n_scen, void* stream);
int gelato_eval_mesh_error_intervals(GelatoPlan* plan, const double* x, double* err_int, int32_t n_scen);
int gelato_eval_mesh_error_intervals_dev(GelatoPlan* plan, const double* x_dev, double* err_int_dev, int32_t n_scen,
                                         void* stream);

/* Path check (DESIGN.md section 11): do the aero constraints (ineqcon_alpha, ineqcon_q, ineqcon_qalpha) hold BETWEEN the
 * nodes?  The NLP enforces them at the state nodes only.  On the grid of gelato_plan_set_mesh_grid, for scenario s and
 * aero job j of the plan (section i, limit L), at each test point l of section i:
 *     v_l = position | velocity | quaternion interpolated with the grid's P row (the chains of the mesh error estimate)
 *     t_l = tau_t[l] (tf - to) / 2 + (tf + to) / 2,   to = t[i], tf = t[i + 1]
 *     r_l = 1 - f(v_l, t_l) / L
 * with f exactly the function objfunc's row of the job evaluates at a node (pristine x, the scenario's units and wind
 * table); res[s][j] = min_l r_l and at[s][j] = the l of the minimum (ties: the smallest l; a NaN is the minimum, the
 * first NaN's l, as numpy.min / numpy.argmin).  A job with range "initial" (one row) is a point constraint with
 * nothing between nodes: res = +inf, at = -1.  Min and 1 - f are exact, so the result has one value.  At a test point
 * that is an LGR node, r_l is objfunc's row for that node bit for bit.
 * res and at are [n_scen][n_aero], in the plan's aero-job order; a plan without aero jobs writes nothing.
 * gelato_eval_path_check: host buffers (page-locked ones are DMA'd directly, others staged).  _dev: device pointers,
 * enqueued on `stream` (NULL = the plan's own), not synchronised.  Both use the scenario blocks, refuse an n_scen beyond
 * them and refuse calls before a grid is set.  Two launches per call (DESIGN.md section 11 gives the measured cost); the
 * _dev call uses plan-owned scratch (n_scen x the test points of the jobs over a whole section doubles): calls on one
 * plan must not overlap on different streams. */
int gelato_eval_path_check(GelatoPlan* plan, const double* x, double* res, int32_t* at, int32_t n_scen);
int gelato_eval_path_check_dev(GelatoPlan* plan, const double* x_dev, double* res_dev, int32_t* at_dev, int32_t n_scen,
                               void* stream);

/* Path rows (DESIGN.md section 11): the aero constraints as inequality rows of the NLP at the test points of a grid of
 * their own, set per plan (separate from the grid of gelato_plan_set_mesh_grid, so re-gridding a diagnosis does not
 * change the NLP).  Opt-in: a plan without path rows evaluates nothing new.
 * Rows: the plan's aero jobs over a whole section (range "all"), in aero-job order, each job's test points l ascending,
 * except a test point whose P row is exactly a unit vector (a support point: that node's own row already holds the
 * constraint there; on the default grid of n + 1 flipped LGR points that drops +1).
 * Value: r = 1 - f(v_l, tn_l) / L, exactly the path check's residual at that test point (same interpolation, time,
 * units and wind table), bit for bit.
 * Jacobian, by the chain rule through the interpolation (the NLP's node rows follow the reference's perturbation
 * protocol; these rows have no reference counterpart):
 *     gq_c = -fd_div(f(v_l + dx e_c, tn_l) - f(v_l, tn_l), dx)   for the 10 state components c (position 3 |
 *            velocity 3 | quaternion 4; max-q rows have no quaternion entries); entry of state row xa + m: P[l][m] gq_c
 *     gq_to / gq_tf: the same with tn_l at to + dx / tf + dx and v_l unchanged; one entry each
 * with dx the plan's dx in forward mode; in central mode (gelato_plan_set_fd, DESIGN.md H6) every quotient is
 * fd_central(gq(+h), gq(-h)).  The entries follow the mode at launch.
 * Values of one scenario, variable-major (each funcsSens block a contiguous range): position, 3 (n + 1) per row in
 * (m, c) order, rows in list order | velocity, the same | quaternion, 4 (n + 1) per row of kinds alpha and Q-alpha |
 * t, (to, tf) per row.
 * gelato_plan_set_path_rows: the grid as gelato_plan_set_mesh_grid takes it, with the same checks and reasons; a
 * refused grid leaves the plan unchanged.
 * gelato_plan_path_rows: *n_rows, *n_vals (values per scenario) and, per row, its aero job, test point and the offsets
 * off[row][4] (position | velocity | quaternion (-1: none) | t) of its entries; job / l / off may be NULL.
 * gelato_eval_path_rows: g_path[n_scen][n_rows] and vals_path[n_scen][n_vals] of x[n_scen][n_vars]; either may be NULL
 * (g_path only: the centre evaluations alone).  Host buffers as gelato_eval_path_check; _dev: device pointers on
 * `stream` (NULL = the plan's own), not synchronised.  Both use the scenario blocks and refuse an n_scen beyond them,
 * refuse calls before path rows are set, and write nothing for a plan with zero rows.  One launch (k_path_rows). */
int gelato_plan_set_path_rows(GelatoPlan* plan, const GelatoMeshGridDesc* grid);
int gelato_plan_path_rows(const GelatoPlan* plan, int32_t* n_rows, int64_t* n_vals, int32_t* job, int32_t* l, int64_t* off);
int gelato_eval_path_rows(GelatoPlan* plan, const double* x, double* g_path, double* vals_path, int32_t n_scen);
int gelato_eval_path_rows_dev(GelatoPlan* plan, const double* x_dev, double* g_dev, double* vals_dev, int32_t n_scen,
                              void* stream);

int gelato_host_alloc(size_t bytes, void** out);
int gelato_host_free(void* ptr);

/* Device-resident entry points: pointers are device memory, work is enqueued on
 * `stream` (a cudaStream_t, NULL = the plan's own stream) and NOT synchronised.
 * A vals_dev buffer must be initialised ONCE with gelato_fill_template (constants and
 * D entries, which never change); gelato_eval_jacobian_dev then rewrites every
 * x-dependent slot on each call and leaves the constants alone. */
int gelato_eval_residuals_dev(GelatoPlan* plan, const double* x_dev, double* g_dev, int32_t n_scen, void* stream);
int gelato_fill_template(GelatoPlan* plan, double* vals_dev, int32_t n_scen, void* stream);
/* objfunc + sens of the same x_dev as ONE launch of the Jacobian kernel: its dynamics blocks already hold the
 * right-hand side at the pristine x (their centre column) and write the collocation defects (D.X computed by
 * otherwise idle threads of phase 0) next to the Jacobian values; aero and event blocks carry one more column at
 * the pristine state; the linear rows and the objective are blocks of their own.  Bit-identical to the two
 * separate calls.
 * _packed_dev: the same with the packed Jacobian output ([n_scen][n_pack], see gelato_eval_pair_packed). */
int gelato_eval_pair_dev(GelatoPlan* plan, const double* x_dev, double* g_dev, double* vals_dev, int32_t n_scen,
                         void* stream);
int gelato_eval_pair_packed_dev(GelatoPlan* plan, const double* x_dev, double* g_dev, double* packed_dev, int32_t n_scen,
                                void* stream);
/* ONE problem sharded over GPUs (SURVEY.md 8(e)-2): the pair evaluation restricted to blocks [block_first, block_first +
 * block_count) of the plan's block table (gelato_plan_n_blocks(plan, 4) blocks: dynamics, aero rows, event rows,
 * linear rows) and vacuum dynamics nodes [vac_first, vac_first + vac_count) (gelato_plan_n_blocks(plan, 5) nodes).
 * Every packed slot and residual row is written by exactly one block or node: ranks with disjoint covering ranges
 * fill disjoint parts of packed[] and g[] (gelato_b200/batch.py: ShardedProblem finds each rank's part once and
 * gathers).  The result-table user constraints (GT_*) are evaluated by the range that starts at block 0 (block_first ==
 * 0, block_count > 0), in full.  Device pointers, caller's stream, not synchronised.  Forward differences only: in
 * central mode it returns GELATO_ERR_ARG. */
int gelato_eval_pair_packed_range_dev(GelatoPlan* plan, const double* x_dev, double* g_dev, double* packed_dev, int32_t n_scen,
                                      int32_t block_first, int32_t block_count, int32_t vac_first, int32_t vac_count,
                                      void* stream);

int gelato_eval_jacobian_dev(GelatoPlan* plan, const double* x_dev, double* vals_dev, int32_t n_scen, void* stream);
/* packed_dev[n_scen][n_xdep] = the x-dependent slots of vals_dev[n_scen][n_vals], in ascending slot order */
int gelato_pack_xdep_dev(GelatoPlan* plan, const double* vals_dev, double* packed_dev, int32_t n_scen, void* stream);

/* Timing helper for benchmarks: runs `reps` back-to-back launches of the chosen kernel on device-resident
 * buffers and returns the average duration in milliseconds measured with CUDA events on the launch stream.
 * which: 0 residual kernel | 1 the Jacobian kernel | 2 the heavy roles' blocks alone (air dynamics + aero rows)
 * | 3 the light roles' blocks alone (vacuum dynamics, fallback, event rows).  Always forward differences with the
 * plan's dx, whatever gelato_plan_set_fd chose (this and gelato_launch_kernel_dev time the kernels themselves). */
int gelato_time_kernel(GelatoPlan* plan, int which, const double* x_dev, double* out_dev, int32_t n_scen, int reps,
                       float* avg_ms);
/* Measurement helper: enqueue exactly one kernel on `stream`, not synchronised -- for benchmarks that bracket single
 * kernels with their own CUDA events.  which: 0 the residual kernel (out_dev is g) | 1 the Jacobian kernel | 2 / 3 its
 * heavy / light roles' blocks alone (role-subset builds of the same kernel); COO (packed = 0) or packed Jacobian
 * output; g_dev != NULL: as a pair evaluation runs it (objfunc's rows written too). */
int gelato_launch_kernel_dev(GelatoPlan* plan, int which, const double* x_dev, double* out_dev, double* g_dev,
                             int32_t n_scen, int32_t packed, void* stream);

/* 1 if the library was compiled with unfused multiply-add on the device (the
 * build contract, checked by running a probe kernel); 0 otherwise. */
int gelato_selftest_unfused(int device, int* ok);

/* FP64 issue-rate probe (DESIGN.md H9): measured DFMA and DADD+DMUL TFLOP/s. */
int gelato_fp64_peak(int device, double* tflops_fma, double* tflops_nofma);

/* ---- leaf batch entry points ------------------------------------------------------------
 * The reference's pybind11 leaf functions evaluated for n nodes by one kernel launch (one thread per
 * node; same device functions as the fused kernels).  Host buffers in and out, row-major, synchronous.
 * They replace, argument for argument:
 *   gelato_leaf_dynamics_velocity        dynamics_c.dynamics_velocity(mass_e, pos, vel, quat, t, param, wind, CA, units)
 *                                         (/root/reference/src/pybind_dynamics.cpp:30-71; param[5], units[3]; out n x 3)
 *   gelato_leaf_dynamics_velocity_noair  dynamics_c.dynamics_velocity_NoAir (:73-92)
 *   gelato_leaf_dynamics_quaternion      dynamics_c.dynamics_quaternion (:94-106; out n x 4)
 *   gelato_leaf_aero                     utils_c.angle_of_attack_all_array_rad (kind 0), dynamic_pressure_array_pa
 *                                         (kind 1, quat may be NULL), q_alpha_array_pa_rad (kind 2),
 *                                         angle_of_attack_ab_array_rad (kind 3, out n x 2: pitch-plane, yaw-plane),
 *                                         wind_ned (kind 4: t[] carries the altitudes, pos / vel / quat unused, out n x 3)
 *                                         (/root/reference/src/wrapper_utils.hpp:82-206; dimensional inputs, t in seconds)
 *   gelato_leaf_eci2geodetic             coordinate_c.eci2geodetic (wrapper_coordinate.hpp:193-199; lat deg, lon deg, alt m)
 *   gelato_leaf_gravity                  coordinate_c.gravity (gravity.cpp:11-57)
 *   gelato_leaf_iip                      IIP_c.posLLH_IIP_FAA(posECEF, velECEF, fill_na) (pybind_IIP.cpp:34-51)
 *   gelato_leaf_atmosphere               USStandardAtmosphere_c: out[i] = geopotential_altitude, airtemperature_at,
 *                                         airpressure_at, airdensity_at, speed_of_sound of altitude[i] (n x 5)
 */
int gelato_leaf_dynamics_velocity(int device, int32_t n, const double* mass_e, const double* pos_e,
                                  const double* vel_e, const double* quat, const double* t, const double* param5,
                                  const double* wind, int32_t n_wind, const double* ca, int32_t n_ca,
                                  const double* units3, double* out);
int gelato_leaf_dynamics_velocity_noair(int device, int32_t n, const double* mass_e, const double* pos_e,
                                        const double* quat, const double* param5, const double* units3, double* out);
int gelato_leaf_dynamics_quaternion(int device, int32_t n, const double* quat, const double* u_e, double unit_u,
                                    double* out);
int gelato_leaf_aero(int device, int32_t kind, int32_t n, const double* pos, const double* vel, const double* quat,
                     const double* t, const double* wind, int32_t n_wind, double* out);
int gelato_leaf_eci2geodetic(int device, int32_t n, const double* pos_eci, const double* t, double* out);
int gelato_leaf_gravity(int device, int32_t n, const double* pos_eci, double* out);
int gelato_leaf_iip(int device, int32_t n, const double* pos_ecef, const double* vel_ecef, int32_t fill_na,
                    double* out);
int gelato_leaf_atmosphere(int device, int32_t n, const double* altitude, double* out);

/* The numeric body of the reference's result table (/root/reference/output_result.py:130-261) for n state
 * nodes (any number of solved trajectories concatenated): one thread per node computes the 34 derived
 * quantities the reference obtains through ~30 leaf calls per node.  Inputs dimensional (kg, m, m/s), t in
 * seconds, quat as stored in the decision vector (normalised inside), per-node thrust_vac / air_area /
 * nozzle_area of the section the reference attributes the node to.  out is [n][34] in the order
 *   thrust, lat, lon, lat_IIP, lon_IIP, downrange, altitude, altitude_apogee, altitude_perigee, inclination,
 *   argument_perigee, lon_ascending_node, true_anomaly, vel_ground_NED_X/Y/Z, accel_BODY_X, aero_BODY_X,
 *   heading/pitch/roll_NED2BODY, flightpath, azimuth (inertial velocity, geocentric), thrust_direction_ECI_X/Y/Z,
 *   vel_ground, vel_air, AOA_total, AOA_pitch, AOA_yaw, dynamic_pressure, Q_alpha, M
 * (gelato_b200/output.py assembles the reference's DataFrame columns from it). */
int gelato_leaf_output_table(int device, int32_t n, const double* mass, const double* pos, const double* vel,
                             const double* quat, const double* t, const double* thrust_vac, const double* air_area,
                             const double* nozzle_area, const double* wind, int32_t n_wind, const double* ca, int32_t n_ca,
                             double launch_lat_deg, double launch_lon_deg, double* out);

/* The forward-simulation initial guess (/root/reference/initialize.py:114-179 rocket_simulation with :37-111
 * dynamics_init, :182-221 zerolift_turn_correct and :229-235 integrate_runge_kutta_4d) for n scenarios at once,
 * ONE THREAD PER SCENARIO: classical Runge-Kutta from t_init to t_out[n_out-1] in steps of dt through the event
 * schedule, then the states interpolated (numpy.interp) at t_out.  The reference runs it once per settings file in
 * Python (its dt = 0.005 s: about half a million right-hand sides); a dispersed study needs one per scenario.
 *   x_init            11 values per scenario: mass, position[3], velocity[3], quaternion[4] (dimensional)
 *   events            n_ev rows per scenario of {time, thrust, massflow, reference_area, nozzle_area, mass_jettison}
 *                     (pdict["params"][i]; times ascending)
 *   zlt               n_ev flags: the event's attitude is "zero-lift-turn" (shared by the scenarios)
 *   u_table           n_u rows {time, roll, pitch, yaw rate [deg/s]} (shared)
 *   wind, ca          the tables of gelato_leaf_dynamics_velocity
 *   scenario_strides  4 values: doubles between consecutive scenarios of x_init, events, wind, ca; 0 = every
 *                     scenario reads the one copy given
 *   x_out             [n][n_out][11]
 *   u_out             [n][n_out][3] or NULL: the reference's second return value (the rate history at t_out)
 * Same results as the reference's function bit for bit with its libm replaced by gmath.h (tests/test_initguess.py). */
int gelato_init_rocket_simulation(int device, int32_t n, const double* x_init, const double* events, const int32_t* zlt,
                                  int32_t n_ev, const double* u_table, int32_t n_u, const double* wind, int32_t n_wind,
                                  const double* ca, int32_t n_ca, const int64_t* scenario_strides, double t_init,
                                  const double* t_out, int32_t n_out, double dt, double* x_out, double* u_out);

/* The coordinate_c leaves that are not on the NLP path (/root/reference/src/pybind_coordinate.cpp:28-78), n items by
 * one launch, one thread per item.  fn: GC_* below; a / b: per-item input vectors of a_width / b_width doubles (0..9);
 * t: per-item time or NULL; out: [n][width of the function's result].
 *   code  function (reference name)            a                      b            t   out
 *    0    quatmult                             q[4]                   p[4]             4
 *    1    conj                                 q[4]                                    4
 *    2/3  normalize (3 / 4 elements)           v                                       3 / 4
 *    4    quatrot                              q[4]                   v[3]             3
 *    5    ecef2geodetic                        x, y, z                                 lat deg, lon deg, alt m
 *    6    geodetic2ecef                        lat deg, lon deg, alt                   3
 *    7/8  ecef2eci / eci2ecef                  v[3]                                t   3
 *    9/10 vel_ecef2eci / vel_eci2ecef          vel[3]                 pos[3]       t   3
 *   11/12 quat_eci2ecef / quat_ecef2eci                                            t   4
 *   13/14 quat_ecef2nedg / quat_nedg2ecef      pos_ecef[3]                             4
 *   15/16 quat_eci2nedg / quat_nedg2eci        pos_eci[3]                          t   4
 *   17    quat_from_euler                      az, el, ro deg                          4
 *   18    euler_from_quat                      q[4]                                    3 (deg)
 *   19    quat_nedg2body                       quat_eci2body[4]       pos_eci[3]   t   4
 *   20    orbital_elements                     pos[3]                 vel[3]           a, e, i, Omega, omega, nu (deg)
 *   21    distance_vincenty                    lat0, lon0, lat1, lon1 deg              1 (m)
 *   22-26 angular_momentum_vec, angular_momentum, inclination_rad, inclination_cosine, orbit_energy
 *                                              pos[3]                 vel[3]           3 / 1 / 1 / 1 / 1
 *   27/28 angular_momentum_from_altitude / orbit_energy_from_altitude   ha, hp         1
 *   29 laplace_vector (pybind_coordinate.cpp:70)  pos[3]                 vel[3]           3
 *   30 haversine (utils_c, pybind_utils.cpp:29)   lon1, lat1, lon2, lat2 (deg)            r         1
 *   31 dcm_from_quat (:33)                        q[4]                                              9 (row-major C)
 *   32/33 quat_from_dcm (:35) / euler_from_dcm (:53, degrees)   C[9] row-major                     4 / 3
 *   34 dcm_from_thrustvector (:55)                pos_eci[3]             thrustvec_eci[3]           9
 * Widths: a and b up to 9 values per item, up to 9 outputs. */
enum {
  GC_QUATMULT = 0, GC_CONJ, GC_NORMALIZE3, GC_NORMALIZE4, GC_QUATROT, GC_ECEF2GEODETIC, GC_GEODETIC2ECEF, GC_ECEF2ECI,
  GC_ECI2ECEF, GC_VEL_ECEF2ECI, GC_VEL_ECI2ECEF, GC_QUAT_ECI2ECEF, GC_QUAT_ECEF2ECI, GC_QUAT_ECEF2NEDG, GC_QUAT_NEDG2ECEF,
  GC_QUAT_ECI2NEDG, GC_QUAT_NEDG2ECI, GC_QUAT_FROM_EULER, GC_EULER_FROM_QUAT, GC_QUAT_NEDG2BODY, GC_ORBITAL_ELEMENTS,
  GC_DISTANCE_VINCENTY, GC_ANGMOM_VEC, GC_ANGMOM, GC_INCLINATION_RAD, GC_INCLINATION_COS, GC_ORBIT_ENERGY,
  GC_ANGMOM_FROM_ALT, GC_ENERGY_FROM_ALT, GC_LAPLACE_VECTOR, GC_HAVERSINE, GC_DCM_FROM_QUAT, GC_QUAT_FROM_DCM,
  GC_EULER_FROM_DCM, GC_DCM_FROM_THRUSTVECTOR, GC_N_FUNCTIONS
};
int gelato_leaf_coordinate(int device, int32_t fn, int32_t n, const double* a, int32_t a_width, const double* b, int32_t b_width,
                           const double* t, double* out);

#ifdef __cplusplus
}
#endif
#endif /* GELATO_B200_H_ */
