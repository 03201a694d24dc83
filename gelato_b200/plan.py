"""Problem compiler: (pdict, unitdict, condition) -> flat tables for the CUDA engine.

Host side, runs once per problem (and once per dispersed scenario).  It walks the
problem dictionaries exactly as the reference's constraint modules do
(/root/reference/lib/con_dynamics.py, con_aero.py, con_waypoint.py,
con_init_terminal_knot.py, con_trajectory.py, con_user.py, cost_gradient.py) and
emits

  * the row layout of the residual vector g: g[0] = objective, then the 22
    constraint groups in the reference's `funcs` order
    (/root/reference/Trajectory_Optimization.py:194-242);
  * the COO (row, col) int32 arrays of every Jacobian block in the reference's
    exact emission order (the sparsity IPOPT is given once and for all,
    Trajectory_Optimization.py:400-416), and for each block its offset into the
    flat `vals` vector the Jacobian kernel fills;
  * `vals_template`: every value that does not depend on x (D entries, +-1, unit
    constants), which the kernel's output starts from;
  * the section / linear-row / aero-job / event-job tables of
    include/gelato_b200.h, including the perturb-and-restore residue counts the
    reference's in-place finite differences leave behind (SURVEY.md A.4 / H3).

Nothing here evaluates physics; the numbers the solver sees all come from the
CUDA kernels.
"""
import math

import numpy as np

from . import hostmath
from .output import KERNEL_COLUMNS

EQ_GROUPS = (
    "eqcon_init eqcon_time eqcon_dyn_mass eqcon_dyn_pos eqcon_dyn_vel eqcon_dyn_quat eqcon_knot "
    "eqcon_terminal eqcon_rate eqcon_pos eqcon_iip eqcon_user"
).split()
INEQ_GROUPS = (
    "ineqcon_alpha ineqcon_q ineqcon_qalpha ineqcon_mass ineqcon_kick ineqcon_time ineqcon_pos "
    "ineqcon_iip ineqcon_antenna ineqcon_user"
).split()
GROUPS = EQ_GROUPS + INEQ_GROUPS
VAR_ORDER = ("mass", "position", "velocity", "quaternion", "u", "t")

# include/gelato_b200.h enums
GS_N, GS_UA, GS_XA, GS_FLAGS, GS_D_OFF, GS_TAU_OFF, GS_R_MASS, GS_R_POS, GS_R_VEL, GS_R_QUAT, GS_I32_COLS = range(11)
GSF_ENGINE_ON, GSF_AIR, GSF_AIR_FD, GSF_HOLD = 1, 2, 4, 8
(GS_JP_VEL, GS_JP_T, GS_JV_MASS, GS_JV_POS, GS_JV_VEL, GS_JV_QUAT, GS_JV_T, GS_JQ_QUAT, GS_JQ_U, GS_JQ_T,
 GS_I64_COLS) = range(11)
GS_THRUST, GS_MASSFLOW, GS_REF_AREA, GS_NOZZLE_AREA, GS_F64_COLS = range(5)
GL_ROW, GL_IDX_PLUS, GL_IDX_MINUS, GL_I32_COLS = range(4)
GL_SCALE_PLUS, GL_SCALE_MINUS, GL_CONST, GL_F64_COLS = range(4)
GA_KIND, GA_SECTION, GA_NK, GA_ROW0, GA_I32_COLS = range(5)
GA_J_POS, GA_J_VEL, GA_J_QUAT, GA_J_T, GA_I64_COLS = range(5)
GA_LIMIT, GA_F64_COLS = range(2)
GE_LLH, GE_IIP, GE_ANT, GE_TERM, GE_USER_ORBIT = range(5)
GE_USER_PERIGEE = GE_USER_ORBIT
GE_TYPE, GE_TIDX, GE_SROW, GE_COMP, GE_FORM, GE_ROW, GE_NROW, GE_RC0 = range(8)
GE_I32_COLS = GE_RC0 + 7
(GEF_DIFF_OVER_DEN, GEF_NEG_DIFF_OVER_DEN, GEF_RATIO_M1, GEF_NEG_RATIO_P1, GEF_REF_MINUS_OVER_DEN,
 GEF_MINUS_REF) = range(6)
GE_J_POS, GE_J_VEL, GE_J_T, GE_I64_COLS = range(4)
GE_REF, GE_DEN, GE_A0, GE_A1, GE_A2, GE_A3, GE_A4, GE_A5, GE_F64_COLS = range(9)

AUX_PER_USER = 12  # per row: 6 finite differences + 6 "background" quotients (jobs.h, GE_USER_ORBIT)
# include/gelato_b200.h: result-table jobs (GT_*)
GT_SROW, GT_TIDX, GT_ROW, GT_NROW, GT_R0, GT_RC0 = range(6)
GT_I32_COLS = GT_RC0 + 12
AUX_PER_TABLE = 18  # per row: 12 finite differences + background quotients after 1, 4, 7, 11, 12 and 0 restores
TABLE_COLUMNS = {name: k for k, name in enumerate(KERNEL_COLUMNS)}  # column codes: output.h / gelato_leaf_output_table
# the slot of a table row's aux values holding the background quotient after k restores (user_table.h)
_TABLE_BG_SLOT = {1: 12, 4: 13, 7: 14, 11: 15, 12: 16, 0: 17}

# quantity codes of the user built-ins (include/gelato_b200.h: GEQ_*)
ORBIT_QUANTITIES = {"perigee_radius": 0, "apogee_radius": 1, "semi_major_axis": 2, "eccentricity": 3,
                    "inclination_deg": 4, "orbit_energy": 5, "angular_momentum": 6}


class _UserBlocks(dict):
    """{variable: (rows, size) array} of one user-constraint group; the arrays are column slices of `buffer`."""

    def __init__(self, buffer):
        super().__init__()
        self.buffer = buffer


class OrbitAtEvent:
    """GPU-resident built-in user constraint (the registry the reference's `user_constraints.py` hook maps onto,
    /root/reference/lib/con_user.py:33-42): up to three rows

        g_r = quantity_r(position, velocity at the first node of `event_name`) / scale_r - offset_r

    with quantity_r one of ORBIT_QUANTITIES -- the orbital elements and orbit integrals the reference exposes to
    user constraints (`lib.coordinate_c.orbital_elements`, `orbit_energy`, `angular_momentum`;
    example/user_constraints.py:96-139 is `perigee_radius / 6378137 - 1`).  One row returns a scalar, like the
    shipped example; several return a vector, and `jac_fd`'s dense blocks get one line per row."""

    def __init__(self, event_name, rows):
        self.event_name = event_name
        self.rows = [(str(q), float(scale), float(offset)) for q, scale, offset in rows]
        if not 1 <= len(self.rows) <= 3:
            raise ValueError("a built-in user constraint has one to three rows")
        for q, scale, _ in self.rows:
            if q not in ORBIT_QUANTITIES:
                raise ValueError("unknown quantity %r (known: %s)" % (q, ", ".join(sorted(ORBIT_QUANTITIES))))
            if scale == 0.0:
                raise ValueError("scale must be non-zero")


class PerigeeAtEvent(OrbitAtEvent):
    """The shipped example's user constraint (/root/reference/example/user_constraints.py:120-139): perigee radius
    ratio a(1-e)/6378137 - 1 of the state at the first node of a named event."""

    def __init__(self, event_name):
        super().__init__(event_name, [("perigee_radius", 6378137.0, 1.0)])


class TableAtEvent:
    """GPU-resident built-in user constraint on the result table: rows

        g_r = column_r(state at the first node of `event_name`) / scale_r - offset_r

    with column_r one of output.KERNEL_COLUMNS -- the per-node quantities of the reference's result table
    (output_result.py), in its units (deg, m, Pa, m/s, N): altitude, downrange, dynamic_pressure, AOA_total,
    flightpath_vel_inertial_geocentric, ...  The node is the one OrbitAtEvent uses; its inputs are those the result table
    gives that node: mass, position, velocity, quaternion, time t[i] * unit_t, section i's thrust / reference_area /
    nozzle_area, the wind and CA tables and the launch site.  One row returns a scalar; several return a vector.
    A user group may also be a list of built-ins (OrbitAtEvent and TableAtEvent mixed): their rows in list order."""

    def __init__(self, event_name, rows):
        self.event_name = event_name
        self.rows = [(str(col), float(scale), float(offset)) for col, scale, offset in rows]
        if not self.rows:
            raise ValueError("a built-in user constraint has at least one row")
        for col, scale, _ in self.rows:
            if col not in TABLE_COLUMNS:
                raise ValueError("unknown result-table column %r (known: %s)" % (col, ", ".join(KERNEL_COLUMNS)))
            if scale == 0.0:
                raise ValueError("scale must be non-zero")


def _builtins(fn):
    """The built-ins of a user group: [] for None, the list for a list / tuple, else [fn]; TypeError for anything that
    is not a registered built-in."""
    if fn is None:
        return []
    items = list(fn) if isinstance(fn, (list, tuple)) else [fn]
    if not items or not all(isinstance(b, (OrbitAtEvent, TableAtEvent)) for b in items):
        raise TypeError(
            "user constraints evaluated on the GPU must be registered built-ins (OrbitAtEvent / PerigeeAtEvent, "
            "TableAtEvent) or a non-empty list of them; arbitrary Python callables cannot run inside the CUDA kernels")
    return items


class Block:
    """One (group, variable) COO block of the Jacobian."""

    __slots__ = ("offset", "rows", "cols", "shape")

    def __init__(self, offset, rows, cols, shape):
        self.offset = int(offset)
        self.rows = np.ascontiguousarray(rows, dtype="i4")
        self.cols = np.ascontiguousarray(cols, dtype="i4")
        self.shape = tuple(int(s) for s in shape)

    @property
    def nnz(self):
        return self.rows.size


def _i4(parts):
    if len(parts) == 0:
        return np.zeros(0, dtype="i4")
    return np.concatenate([np.asarray(p, dtype="i4").ravel() for p in parts])


def _f8(parts):
    if len(parts) == 0:
        return np.zeros(0, dtype="f8")
    return np.concatenate([np.asarray(p, dtype="f8").ravel() for p in parts])


class CompiledPlan:
    """Everything the C ABI's GelatoPlanDesc needs, plus the host-side layout
    used to slice g / vals back into the reference's dictionaries."""

    def __init__(self, pdict, unitdict, condition, user_eq=None, user_ineq=None, coord=None):
        self.p, self.u, self.c = pdict, unitdict, condition
        self.coord = coord or hostmath
        self.ps = pdict["ps_params"]
        self.S = S = int(pdict["num_sections"])
        self.N = N = int(pdict["N"])
        self.M = M = int(pdict["M"])
        self.dx = float(pdict["dx"])
        self.payload_mode = 1 if condition["OptimizationMode"] == "Payload" else 0
        self.sizes = {"mass": M, "position": 3 * M, "velocity": 3 * M, "quaternion": 4 * M, "u": 2 * N, "t": S + 1}
        self.off = {}
        o = 0
        for k in VAR_ORDER:
            self.off[k] = o
            o += self.sizes[k]
        self.n_vars = o
        for fn in (user_eq, user_ineq):
            _builtins(fn)
        self.user_eq, self.user_ineq = user_eq, user_ineq

        self._sec = [self.ps.get_index(i) for i in range(S)]
        self._names = [prm["name"] for prm in pdict["params"]]
        self._lin = []  # (row, ip, im, sp, sm, c)
        self._evt = []  # dict per job
        self._tab = []  # dict per result-table job
        self._tab_rows = []  # (column code, scale, offset, aux offset) per result-table row
        self._aero = []
        self.group_rows = {}  # key -> (row0, nrow) | None
        self.blocks = {}  # key -> {var: Block} | None | ("dense-user", ...) (_g_user)
        self._tmpl = []  # (offset, values) constant segments
        self._nvals = 0
        self._row = 1  # g[0] = objective
        self._rc = np.zeros(self.n_vars, dtype=np.int64)

        self._build_sections_static()
        self._compile_groups()
        self._finish()

    # ------------------------------------------------------------------
    def _param(self, i):
        prm = self.p["params"][i]
        return prm["thrust"], prm["massflow"], prm["reference_area"], prm["nozzle_area"]

    def _holds(self, i):
        return self.p["params"][i]["attitude"] in ["hold", "vertical"]

    def _build_sections_static(self):
        S = self.S
        self.sec_i32 = np.zeros((S, GS_I32_COLS), dtype=np.int32)
        self.sec_i64 = np.full((S, GS_I64_COLS), -1, dtype=np.int64)
        self.sec_f64 = np.zeros((S, GS_F64_COLS), dtype=np.float64)
        d_parts, tau_parts = [], []
        d_off = tau_off = 0
        for i in range(S):
            ua, ub, xa, xb, n = self._sec[i]
            thrust, massflow, ref_area, noz = self._param(i)
            flags = 0
            if self.p["params"][i]["engineOn"]:
                flags |= GSF_ENGINE_ON
            if ref_area != 0.0:
                flags |= GSF_AIR
            if ref_area > 0.0:
                flags |= GSF_AIR_FD
            if self._holds(i):
                flags |= GSF_HOLD
            self.sec_i32[i, [GS_N, GS_UA, GS_XA, GS_FLAGS, GS_D_OFF, GS_TAU_OFF]] = [n, ua, xa, flags, d_off, tau_off]
            self.sec_f64[i] = [thrust, massflow, ref_area, noz]
            D = np.ascontiguousarray(self.ps.D(i), dtype=np.float64)
            d_parts.append(D.ravel())
            tau_parts.append(np.asarray(self.ps.tau(i), dtype=np.float64))
            d_off += D.size
            tau_off += n
        self.d_pool = _f8(d_parts)
        self.tau_pool = _f8(tau_parts)

    # ------------------------------------------------------------------
    # helpers used while walking the groups
    def _begin(self, key, nrow):
        """Reserve rows for a present group; returns its first row in g."""
        row0 = self._row
        self.group_rows[key] = (row0, int(nrow))
        self._row += int(nrow)
        return row0

    def _absent(self, key):
        self.group_rows[key] = None
        self.blocks[key] = None

    def _block(self, key, var, rows, cols, shape, const=None):
        """Append a COO block; `const` (same length) goes to the template."""
        rows = np.asarray(rows).ravel()
        blk = Block(self._nvals, rows, np.asarray(cols).ravel(), shape)
        assert blk.rows.size == blk.cols.size
        if const is not None:
            const = np.asarray(const, dtype=np.float64).ravel()
            assert const.size == blk.nnz, (key, var, const.size, blk.nnz)
            self._tmpl.append((blk.offset, const))
        self.blocks.setdefault(key, {})[var] = blk
        self._nvals += blk.nnz
        return blk

    def _lin_row(self, row, ip, im, c=0.0, sp=1.0, sm=1.0):
        self._lin.append((int(row), -1 if ip is None else int(ip), -1 if im is None else int(im), float(sp),
                          float(sm), float(c)))

    def _x(self, var, idx):
        return self.off[var] + int(idx)

    # ------------------------------------------------------------------
    def _compile_groups(self):
        """Groups in the order objfunc / sens evaluate them
        (Trajectory_Optimization.py:194-312); the order matters for the residue
        bookkeeping (`self._rc`)."""
        self._g_init()
        self._g_time()
        self._g_dyn_mass()
        self._g_dyn_pos()
        self._g_dyn_vel()
        self._g_dyn_quat()
        self._g_knot()
        self._g_terminal()
        self._g_rate()
        self._g_posllh("eqcon_pos", True)
        self._g_iip("eqcon_iip", True)
        self._g_user("eqcon_user", self.user_eq)
        self.rc_aero = np.minimum(self._rc, 255).astype(np.uint8)
        assert self._rc.max() <= 255
        for key, kind in (("ineqcon_alpha", 0), ("ineqcon_q", 1), ("ineqcon_qalpha", 2)):
            self._g_aero(key, kind)
        self._g_ineq_mass()
        self._g_kick()
        self._g_ineq_time()
        self._g_posllh("ineqcon_pos", False)
        self._g_iip("ineqcon_iip", False)
        self._g_antenna()
        self._g_user("ineqcon_user", self.user_ineq)

    # ---- init / time (con_init_terminal_knot.py:41-171) ----------------
    def _g_init(self):
        c, u, M = self.c, self.u, self.M
        off = 0 if self.payload_mode else 1
        nrow = 10 + off
        r0 = self._begin("eqcon_init", nrow)
        if off:
            self._lin_row(r0, self._x("mass", 0), None, -(c["init"]["mass"] / u["mass"]))
            self._block("eqcon_init", "mass", [0], [0], (nrow, M), [1.0])
        init_pos = np.asarray(c["init"]["position"]) / u["position"]
        init_vel = np.asarray(c["init"]["velocity"]) / u["velocity"]
        init_quat = np.asarray(c["init"]["quaternion"], dtype=np.float64)
        for k in range(3):
            self._lin_row(r0 + off + k, self._x("position", k), None, -init_pos[k])
            self._lin_row(r0 + off + 3 + k, self._x("velocity", k), None, -init_vel[k])
        for k in range(4):
            self._lin_row(r0 + off + 6 + k, self._x("quaternion", k), None, -init_quat[k])
        self._block("eqcon_init", "position", np.arange(off, off + 3), np.arange(3), (nrow, M * 3), np.ones(3))
        self._block("eqcon_init", "velocity", np.arange(off + 3, off + 6), np.arange(3), (nrow, M * 3), np.ones(3))
        self._block("eqcon_init", "quaternion", np.arange(off + 6, off + 10), np.arange(4), (nrow, M * 4), np.ones(4))

    def _timed_events(self):
        prm, idx = self.p["params"], self.p["event_index"]
        return [(i, idx[prm[i]["time_ref"]]) for i in range(1, self.S + 1) if prm[i]["time_ref"] in idx]

    def _g_time(self):
        prm, ut = self.p["params"], self.u["t"]
        ev = self._timed_events()
        r0 = self._begin("eqcon_time", len(ev) + 1)
        self._lin_row(r0, self._x("t", 0), None, -(prm[0]["time"] / ut))
        r, c, d = [0], [0], [1.0]
        for k, (i, ir) in enumerate(ev):
            self._lin_row(r0 + 1 + k, self._x("t", i), self._x("t", ir), -((prm[i]["time"] - prm[ir]["time"]) / ut))
            r += [k + 1, k + 1]
            c += [i, ir]
            d += [1.0, -1.0]
        self._block("eqcon_time", "t", r, c, (len(ev) + 1, self.S + 1), d)

    # ---- dynamics (con_dynamics.py) ------------------------------------
    def _g_dyn_mass(self):
        um, ut = self.u["mass"], self.u["t"]
        r0 = self._begin("eqcon_dyn_mass", self.N)
        mr, mc, md, tr, tc, td = [], [], [], [], [], []
        for i in range(self.S):
            ua, ub, xa, xb, n = self._sec[i]
            self.sec_i32[i, GS_R_MASS] = r0 + ua
            if self.p["params"][i]["engineOn"]:
                mr.append(np.repeat(np.arange(ua, ub), n + 1))
                mc.append(np.tile(np.arange(xa, xb), n))
                md.append(self.ps.D(i).ravel(order="C"))
                mf = self.p["params"][i]["massflow"]
                tr += [np.arange(ua, ub), np.arange(ua, ub)]
                tc += [np.full(n, i), np.full(n, i + 1)]
                td += [np.full(n, -mf / um * ut / 2.0), np.full(n, mf / um * ut / 2.0)]
            else:
                mr += [np.arange(ua, ub), np.arange(ua, ub)]
                mc += [np.full(n, xa), np.arange(xa + 1, xb)]
                md += [np.full(n, -1.0), np.full(n, 1.0)]
        self._block("eqcon_dyn_mass", "mass", _i4(mr), _i4(mc), (self.N, self.M), _f8(md))
        self._block("eqcon_dyn_mass", "t", _i4(tr), _i4(tc), (self.N, self.S + 1), _f8(td))

    def _g_dyn_pos(self):
        N3, M3 = self.N * 3, self.M * 3
        r0 = self._begin("eqcon_dyn_pos", N3)
        pr, pc, pd, vr, vc, tr, tc = ([] for _ in range(7))
        for i in range(self.S):
            ua, ub, xa, xb, n = self._sec[i]
            self.sec_i32[i, GS_R_POS] = r0 + 3 * ua
            Di = self.ps.D(i).ravel()
            rows3 = np.arange(ua * 3, ub * 3)
            vr.append(rows3)
            vc.append(np.arange((xa + 1) * 3, xb * 3))
            tr += [rows3, rows3]
            tc += [np.full(n * 3, i), np.full(n * 3, i + 1)]
            for k in range(3):
                pr.append(np.repeat(np.arange(ua * 3 + k, ub * 3 + k, 3), n + 1))
                pc.append(np.tile(np.arange(xa * 3 + k, xb * 3 + k, 3), n))
                pd.append(Di)
        self._block("eqcon_dyn_pos", "position", _i4(pr), _i4(pc), (N3, M3), _f8(pd))
        bv = self._block("eqcon_dyn_pos", "velocity", _i4(vr), _i4(vc), (N3, M3))
        bt = self._block("eqcon_dyn_pos", "t", _i4(tr), _i4(tc), (N3, self.S + 1))
        for i in range(self.S):
            ua = self._sec[i][0]
            self.sec_i64[i, GS_JP_VEL] = bv.offset + 3 * ua
            self.sec_i64[i, GS_JP_T] = bt.offset + 6 * ua

    def _g_dyn_vel(self):
        N3, M = self.N * 3, self.M
        r0 = self._begin("eqcon_dyn_vel", N3)
        acc = {k: ([], []) for k in ("mass", "position", "velocity", "quaternion", "t")}
        vel_tmpl = []
        sizes = {k: [] for k in acc}
        for i in range(self.S):
            ua, ub, xa, xb, n = self._sec[i]
            self.sec_i32[i, GS_R_VEL] = r0 + 3 * ua
            rows_nodes = np.arange(ua * 3, ub * 3)
            xs = np.arange(xa + 1, xb)
            acc["mass"][0].append(rows_nodes)
            acc["mass"][1].append(np.repeat(xs, 3))
            for k in range(3):
                acc["position"][0].append(rows_nodes)
                acc["position"][1].append(np.repeat(xs * 3 + k, 3))
            D = self.ps.D(i)
            zero = np.zeros_like(D)
            for ki in range(3):
                for kj in range(3):
                    acc["velocity"][0].append(np.repeat(np.arange(ua * 3 + ki, ub * 3 + ki, 3), n + 1))
                    acc["velocity"][1].append(np.tile(np.arange(xa * 3 + kj, xb * 3 + kj, 3), n))
                    vel_tmpl.append(D if ki == kj else zero)
            for k in range(4):
                acc["quaternion"][0].append(rows_nodes)
                acc["quaternion"][1].append(np.repeat(xs * 4 + k, 3))
            acc["t"][0].extend([rows_nodes, rows_nodes])
            acc["t"][1].extend([np.full(n * 3, i), np.full(n * 3, i + 1)])
            sizes["mass"].append(3 * n)
            sizes["position"].append(9 * n)
            sizes["velocity"].append(9 * n * (n + 1))
            sizes["quaternion"].append(12 * n)
            sizes["t"].append(6 * n)
            # in-place perturbation of rows xa+1 .. xb-1 (con_dynamics.py:362-449)
            air_fd = bool(self.sec_i32[i, GS_FLAGS] & GSF_AIR_FD)
            self._rc[self.off["mass"] + xs] += 1
            for w, var in ((3, "position"), (4, "quaternion")):
                self._rc[self.off[var] + (xa + 1) * w: self.off[var] + xb * w] += 1
            if air_fd:
                self._rc[self.off["velocity"] + (xa + 1) * 3: self.off["velocity"] + xb * 3] += 1
        shapes = {"mass": (N3, M), "position": (N3, M * 3), "velocity": (N3, M * 3), "quaternion": (N3, M * 4),
                  "t": (N3, self.S + 1)}
        cols = {"mass": GS_JV_MASS, "position": GS_JV_POS, "velocity": GS_JV_VEL, "quaternion": GS_JV_QUAT,
                "t": GS_JV_T}
        for var in ("mass", "position", "velocity", "quaternion", "t"):
            const = _f8(vel_tmpl) if var == "velocity" else None
            blk = self._block("eqcon_dyn_vel", var, _i4(acc[var][0]), _i4(acc[var][1]), shapes[var], const)
            starts = np.concatenate(([0], np.cumsum(sizes[var])[:-1]))
            self.sec_i64[:, cols[var]] = blk.offset + starts

    def _g_dyn_quat(self):
        N4 = self.N * 4
        r0 = self._begin("eqcon_dyn_quat", N4)
        acc = {k: ([], []) for k in ("quaternion", "u", "t")}
        q_tmpl = []
        starts = {k: [] for k in acc}
        pos = {k: 0 for k in acc}
        for i in range(self.S):
            ua, ub, xa, xb, n = self._sec[i]
            self.sec_i32[i, GS_R_QUAT] = r0 + 4 * ua
            rows = np.arange(ua * 4, ub * 4)
            if self._holds(i):
                acc["quaternion"][0].extend([rows, rows])
                acc["quaternion"][1].extend([np.tile(np.arange(xa * 4, (xa + 1) * 4), n), np.arange((xa + 1) * 4, xb * 4)])
                q_tmpl.extend([np.full(4 * n, -1.0), np.full(4 * n, 1.0)])
                pos["quaternion"] += 8 * n
                for k in acc:
                    starts[k].append(-1)
                continue
            D = self.ps.D(i)
            sub = np.zeros((n * 4, (n + 1) * 4))
            for k in range(4):
                sub[k::4, k::4] = D
            for k in acc:
                starts[k].append(pos[k])
            acc["quaternion"][0].append(np.repeat(rows, (n + 1) * 4))
            acc["quaternion"][1].append(np.tile(np.arange(xa * 4, xb * 4), n * 4))
            q_tmpl.append(sub)
            pos["quaternion"] += 16 * n * (n + 1)
            for k in range(2):
                acc["u"][0].append(rows)
                acc["u"][1].append(np.repeat(np.arange(ua, ub) * 2 + k, 4))
            pos["u"] += 8 * n
            acc["t"][0].extend([rows, rows])
            acc["t"][1].extend([np.full(n * 4, i), np.full(n * 4, i + 1)])
            pos["t"] += 8 * n
            # in place on xdict["quaternion"], xdict["u"] (con_dynamics.py:580-613)
            self._rc[self.off["quaternion"] + (xa + 1) * 4: self.off["quaternion"] + xb * 4] += 1
            self._rc[self.off["u"] + ua * 2: self.off["u"] + ub * 2] += 1
        shapes = {"quaternion": (N4, self.M * 4), "u": (N4, self.N * 2), "t": (N4, self.S + 1)}
        cols = {"quaternion": GS_JQ_QUAT, "u": GS_JQ_U, "t": GS_JQ_T}
        for var in ("quaternion", "u", "t"):
            const = _f8(q_tmpl) if var == "quaternion" else None
            blk = self._block("eqcon_dyn_quat", var, _i4(acc[var][0]), _i4(acc[var][1]), shapes[var], const)
            for i in range(self.S):
                if starts[var][i] >= 0:
                    self.sec_i64[i, cols[var]] = blk.offset + starts[var][i]

    # ---- knot (con_init_terminal_knot.py:174-326) ----------------------
    def _stage_sections(self):
        out = []
        for stage in self.p["RocketStage"].values():
            if stage["separation_at"] is not None:
                out.append((self._names.index(stage["ignition_at"]), self._names.index(stage["separation_at"]), stage))
        return out

    def _g_knot(self):
        um = self.u["mass"]
        ps = self.ps
        stages = self._stage_sections()
        sep = [sp for _, sp, _ in stages]
        nrow = len(stages) + sum((0 if i in sep else 1) + 10 for i in range(1, self.S))
        r0 = self._begin("eqcon_knot", nrow)
        acc = {k: ([], [], []) for k in ("mass", "position", "velocity", "quaternion")}
        r = 0
        for ig, sp, stage in stages:
            mass_stage = stage["mass_dry"] + stage["mass_propellant"] + sum(
                [item["mass"] for item in stage["dropMass"].values()])
            a, b = ps.index_start_x(ig), ps.index_start_x(sp)
            self._lin_row(r0 + r, self._x("mass", a), self._x("mass", b), -(mass_stage / um))
            acc["mass"][0].extend([r, r])
            acc["mass"][1].extend([a, b])
            acc["mass"][2].extend([1.0, -1.0])
            r += 1
        for i in range(1, self.S):
            xa = ps.index_start_x(i)
            if i not in sep:
                self._lin_row(r0 + r, self._x("mass", xa), self._x("mass", xa - 1),
                              self.p["params"][i]["mass_jettison"] / um)
                acc["mass"][0].extend([r, r])
                acc["mass"][1].extend([xa - 1, xa])
                acc["mass"][2].extend([-1.0, 1.0])
                r += 1
            for key, w in (("position", 3), ("velocity", 3), ("quaternion", 4)):
                for k in range(w):
                    self._lin_row(r0 + r + k, self._x(key, xa * w + k), self._x(key, (xa - 1) * w + k))
                acc[key][0].extend(list(range(r, r + w)) * 2)
                acc[key][1].extend(list(range((xa - 1) * w, xa * w)) + list(range(xa * w, (xa + 1) * w)))
                acc[key][2].extend([-1.0] * w + [1.0] * w)
                r += w
        assert r == nrow
        M = self.M
        shapes = {"mass": (r, M), "position": (r, M * 3), "velocity": (r, M * 3), "quaternion": (r, M * 4)}
        for k, a in acc.items():
            self._block("eqcon_knot", k, a[0], a[1], shapes[k], a[2])

    # ---- terminal (con_init_terminal_knot.py:329-405) ------------------
    def _g_terminal(self):
        c = self.c
        GMe = 3.986004418e14
        if c["altitude_perigee"] is not None and c["altitude_apogee"] is not None:
            c_t = self.coord.angular_momentum_from_altitude(c["altitude_perigee"], c["altitude_apogee"])
            e_t = self.coord.orbit_energy_from_altitude(c["altitude_perigee"], c["altitude_apogee"])
        else:
            c_t = c["radius"] * c["vel_tangential_geocentric"]
            vf = c["vel_tangential_geocentric"] / math.cos(math.radians(c["flightpath_vel_inertial_geocentric"]))
            e_t = vf**2 / 2.0 - GMe / c["radius"]
        has_inc = c["inclination"] is not None
        nrow = 3 if has_inc else 2
        r0 = self._begin("eqcon_terminal", nrow)
        ncol = self.M * 3
        srow = self.M - 1
        job = self._evt_job(GE_TERM, -1, srow, 0, 0, r0, nrow, ref=0.0, den=1.0,
                            a=(e_t, c_t, math.radians(c["inclination"]) if has_inc else 0.0),
                            perturb=("position", "velocity"))
        for key, col in (("position", GE_J_POS), ("velocity", GE_J_VEL)):
            r, cc = [], []
            for j in range(ncol - 3, ncol):
                r += list(range(nrow))
                cc += [j] * nrow
            blk = self._block("eqcon_terminal", key, r, cc, (nrow, ncol))
            job["i64"][col] = blk.offset

    # ---- rate / mass / kick / time (con_trajectory.py, con_init_terminal_knot.py:408-452)
    def _g_rate(self):
        rows_lin = []  # (minus_col | None, plus_col)
        r, c, d = [], [], []
        row0 = 0

        def block(first_col, cols):
            nonlocal row0
            k = len(cols)
            if first_col is not None:
                r.extend(range(row0, row0 + k))
                c.extend([first_col] * k)
                d.extend([-1.0] * k)
            r.extend(range(row0, row0 + k))
            c.extend(cols)
            d.extend([1.0] * k)
            for cc in cols:
                rows_lin.append((first_col, cc))
            row0 += k

        for i in range(self.S):
            ua, ub, xa, xb, n = self._sec[i]
            att = self.p["params"][i]["attitude"]
            if att in ["hold", "vertical"]:
                block(None, list(range(ua * 2, (ua + n) * 2)))
            elif att in ("kick-turn", "pitch"):
                block(ua * 2, list(range((ua + 1) * 2, (ua + n) * 2, 2)))
                block(None, list(range(ua * 2 + 1, (ua + n) * 2 + 1, 2)))
            elif att == "pitch-yaw":
                block(ua * 2, list(range((ua + 1) * 2, (ua + n) * 2, 2)))
                block(ua * 2 + 1, list(range((ua + 1) * 2 + 1, (ua + n) * 2 + 1, 2)))
            elif att == "same-rate":
                block(ua * 2 - 2, list(range(ua * 2, (ua + n) * 2, 2)))
                block(ua * 2 - 1, list(range(ua * 2 + 1, (ua + n) * 2 + 1, 2)))
            elif att in ("zero-lift-turn", "free"):
                pass
            else:  # con_trajectory.py:201-203
                raise SystemExit("ERROR: UNKNOWN ATTITUDE OPTION! ({})".format(att))
        g0 = self._begin("eqcon_rate", row0)
        for k, (first, col) in enumerate(rows_lin):
            self._lin_row(g0 + k, self._x("u", col), None if first is None else self._x("u", first))
        self._block("eqcon_rate", "u", r, c, (row0, self.N * 2), d)

    def _stage_ig_co(self):
        ps = self.ps
        return [(ps.index_start_x(self._names.index(st["ignition_at"])),
                 ps.index_start_x(self._names.index(st["cutoff_at"])), st) for st in self.p["RocketStage"].values()]

    def _g_ineq_mass(self):
        st = self._stage_ig_co()
        r0 = self._begin("ineqcon_mass", len(st))
        r, c, d = [], [], []
        for k, (ig, co, stage) in enumerate(st):
            d_mass = stage["mass_propellant"]
            if stage["dropMass"] is not None:
                d_mass += sum([item["mass"] for item in stage["dropMass"].values()])
            self._lin_row(r0 + k, self._x("mass", co), self._x("mass", ig), d_mass / self.u["mass"])
            r += [k, k]
            c += [ig, co]
            d += [-1.0, 1.0]
        self._block("ineqcon_mass", "mass", r, c, (len(st), self.M), d)

    def _g_kick(self):
        secs = [i for i in range(self.S - 1) if "kick" in self.p["params"][i]["attitude"]]
        nrow = sum(self._sec[i][4] for i in secs)
        r0 = self._begin("ineqcon_kick", nrow)
        r, c, d = [], [], []
        k = 0
        for i in secs:
            ua, ub, _, _, n = self._sec[i]
            for j in range(n):
                self._lin_row(r0 + k + j, None, self._x("u", (ua + j) * 2), 0.0, 1.0, self.u["u"])
            r.extend(range(k, k + n))
            c.extend(range(ua * 2, ub * 2, 2))
            d.extend([-self.u["u"]] * n)
            k += n
        self._block("ineqcon_kick", "u", r, c, (nrow, 2 * self.N), d)

    def _g_ineq_time(self):
        prm, idx = self.p["params"], self.p["event_index"]
        secs = [i for i in range(self.S) if not (prm[i]["time_ref"] in idx and prm[i + 1]["time_ref"] in idx)]
        r0 = self._begin("ineqcon_time", len(secs))
        r, c, d = [], [], []
        for k, i in enumerate(secs):
            self._lin_row(r0 + k, self._x("t", i + 1), self._x("t", i))
            r += [k, k]
            c += [i, i + 1]
            d += [-1.0, 1.0]
        self._block("ineqcon_time", "t", r, c, (len(secs), self.S + 1), d)

    # ---- aero (con_aero.py) --------------------------------------------
    _AERO_KEYS = {0: ("AOA_max", True, True), 1: ("dynamic_pressure_max", False, False), 2: ("Q_alpha_max", True, True)}

    def _g_aero(self, key, kind):
        ckey, in_rad, has_quat = self._AERO_KEYS[kind]
        secs = []
        for i in range(self.S - 1):
            name = self._names[i]
            if name in self.c[ckey]:
                lim = self.c[ckey][name]["value"]
                if in_rad:
                    lim = lim * np.pi / 180.0
                rng = self.c[ckey][name]["range"]
                if rng == "all":
                    nk = self._sec[i][4] + 1
                elif rng == "initial":
                    nk = 1
                else:
                    continue
                secs.append((i, float(lim), nk))
        nrow = sum(s[2] for s in secs)
        if nrow == 0:
            self._absent(key)
            return
        g0 = self._begin(key, nrow)
        acc = {k: ([], []) for k in ("position", "velocity", "quaternion", "t")}
        jobs = []
        pos = {k: 0 for k in acc}
        r0 = 0
        for i, lim, nk in secs:
            xa = self._sec[i][2]
            rows = np.arange(r0, r0 + nk)
            st = dict(pos)
            for var, w in (("position", 3), ("velocity", 3), ("quaternion", 4)):
                if var == "quaternion" and not has_quat:
                    continue
                for j in range(w):
                    acc[var][0].append(rows)
                    acc[var][1].append(np.arange(xa * w + j, (xa + nk) * w + j, w))
                pos[var] += w * nk
            acc["t"][0].extend([rows, rows])
            acc["t"][1].extend([np.full(nk, i), np.full(nk, i + 1)])
            pos["t"] += 2 * nk
            jobs.append((i, lim, nk, g0 + r0, st))
            r0 += nk
        M = self.M
        shapes = {"position": (nrow, M * 3), "velocity": (nrow, M * 3), "quaternion": (nrow, M * 4),
                  "t": (nrow, self.S + 1)}
        blk = {var: self._block(key, var, _i4(acc[var][0]), _i4(acc[var][1]), shapes[var])
               for var in ("position", "velocity", "quaternion", "t")}
        for i, lim, nk, grow, st in jobs:
            self._aero.append({
                "i32": [kind, i, nk, grow],
                "i64": [blk["position"].offset + st["position"], blk["velocity"].offset + st["velocity"],
                        blk["quaternion"].offset + st["quaternion"] if has_quat else -1, blk["t"].offset + st["t"]],
                "f64": [lim],
            })

    # ---- event-point rows (con_waypoint.py) -----------------------------
    def _evt_job(self, typ, tidx, srow, comp, form, row, nrow, ref, den, a=(0.0, 0.0, 0.0), perturb=()):
        """Register an event job; records the residue counts its inputs carry when
        the reference evaluates its gradient, then accounts for the in-place
        perturbation the gradient itself performs on `perturb` variables."""
        rc = [0] * 7
        for k in range(3):
            rc[k] = int(self._rc[self.off["position"] + 3 * srow + k])
            rc[3 + k] = int(self._rc[self.off["velocity"] + 3 * srow + k])
        if tidx >= 0:
            rc[6] = int(self._rc[self.off["t"] + tidx])
        a = list(a) + [0.0] * (6 - len(a))
        job = {"i32": [typ, tidx, srow, comp, form, row, nrow] + rc, "i64": [-1, -1, -1],
               "f64": [float(ref), float(den)] + [float(v) for v in a[:6]]}
        self._evt.append(job)
        for var in perturb:
            self._rc[self.off[var] + 3 * srow: self.off[var] + 3 * srow + 3] += 1
        return job

    def _wp_sections(self):
        if "waypoint" not in self.c:
            return None
        return [(i, self.c["waypoint"][self._names[i]]) for i in range(self.S - 1)
                if self._names[i] in self.c["waypoint"]]

    @staticmethod
    def _bounds(spec, eq):
        """[(sign, ref)] of one waypoint quantity in the reference's row order."""
        out = []
        if eq:
            if "exact" in spec:
                out.append((+1.0, spec["exact"]))
        else:
            if "min" in spec:
                out.append((+1.0, spec["min"]))
            if "max" in spec:
                out.append((-1.0, spec["max"]))
        return out

    def _g_posllh(self, key, eq):
        secs = self._wp_sections()
        if secs is None:
            self._absent(key)
            return
        rows = []
        for i, wp in secs:
            if "downrange" in wp:
                raise NotImplementedError(
                    "downrange waypoints: the reference emits a malformed COO block for them "
                    "(con_waypoint.py:704,917,934); unsupported")
            for comp, name in ((0, "lat"), (1, "lon"), (2, "altitude")):
                if name in wp:
                    for sgn, ref in self._bounds(wp[name], eq):
                        rows.append((i, comp, name, sgn, ref))
        if not rows:
            self._absent(key)
            return
        nrow = len(rows)
        g0 = self._begin(key, nrow)
        pr, pc, tr, tc = [], [], [], []
        jobs = []
        for r, (i, comp, name, sgn, ref) in enumerate(rows):
            xa = self.ps.index_start_x(i)
            if name == "altitude":
                form, den = (GEF_RATIO_M1 if sgn > 0 else GEF_NEG_RATIO_P1), ref
            else:
                form, den = (GEF_DIFF_OVER_DEN if sgn > 0 else GEF_NEG_DIFF_OVER_DEN), (90.0 if name == "lat" else 180.0)
            jobs.append(self._evt_job(GE_LLH, i, xa, comp, form, g0 + r, 1, ref, den, perturb=("position",)))
            pr += [r] * 3
            pc += list(range(xa * 3, (xa + 1) * 3))
            tr.append(r)
            tc.append(i)
        bp = self._block(key, "position", pr, pc, (nrow, self.M * 3))
        bt = self._block(key, "t", tr, tc, (nrow, self.S + 1))
        for r, job in enumerate(jobs):
            job["i64"][GE_J_POS] = bp.offset + 3 * r
            job["i64"][GE_J_T] = bt.offset + r

    def _g_iip(self, key, eq):
        secs = self._wp_sections()
        if secs is None:
            self._absent(key)
            return
        rows = []
        for i, wp in secs:
            for comp, name, den in ((0, "lat_IIP", 90.0), (1, "lon_IIP", 180.0)):
                if name in wp:
                    for sgn, ref in self._bounds(wp[name], eq):
                        rows.append((i, comp, den, sgn, ref))
        if not rows:
            self._absent(key)
            return
        nrow = len(rows)
        g0 = self._begin(key, nrow)
        acc = {k: ([], []) for k in ("position", "velocity", "t")}
        jobs = []
        for r, (i, comp, den, sgn, ref) in enumerate(rows):
            xa = self.ps.index_start_x(i)
            form = GEF_DIFF_OVER_DEN if sgn > 0 else GEF_REF_MINUS_OVER_DEN
            jobs.append(self._evt_job(GE_IIP, i, xa, comp, form, g0 + r, 1, ref, den, perturb=("position", "velocity")))
            for var in ("position", "velocity"):
                acc[var][0].extend([r] * 3)
                acc[var][1].extend(range(xa * 3, (xa + 1) * 3))
            acc["t"][0].append(r)
            acc["t"][1].append(i)
        shapes = {"position": (nrow, self.M * 3), "velocity": (nrow, self.M * 3), "t": (nrow, self.S + 1)}
        blk = {var: self._block(key, var, acc[var][0], acc[var][1], shapes[var]) for var in ("position", "velocity", "t")}
        for r, job in enumerate(jobs):
            job["i64"][GE_J_POS] = blk["position"].offset + 3 * r
            job["i64"][GE_J_VEL] = blk["velocity"].offset + 3 * r
            job["i64"][GE_J_T] = blk["t"].offset + r

    def _g_antenna(self):
        key = "ineqcon_antenna"
        if "antenna" not in self.c:
            self._absent(key)
            return
        rows = []
        for ant in self.c["antenna"].values():
            p_ant = np.asarray(self.coord.geodetic2ecef(ant["lat"], ant["lon"], ant["altitude"]), dtype=np.float64)
            for i in range(self.S - 1):
                if self._names[i] in ant["elevation_min"]:
                    rows.append((i, p_ant, ant["elevation_min"][self._names[i]]))
        if not rows:
            self._absent(key)
            return
        nrow = len(rows)
        g0 = self._begin(key, nrow)
        pr, pc, tr, tc = [], [], [], []
        jobs = []
        for r, (i, p_ant, el) in enumerate(rows):
            xa = self.ps.index_start_x(i)
            ref = np.sin(el * np.pi / 180.0)
            jobs.append(self._evt_job(GE_ANT, i, xa, 0, GEF_MINUS_REF, g0 + r, 1, ref, 1.0, a=p_ant,
                                      perturb=("position",)))
            pr += [r] * 3
            pc += list(range(xa * 3, (xa + 1) * 3))
            tr.append(r)
            tc.append(i)
        bp = self._block(key, "position", pr, pc, (nrow, self.M * 3))
        bt = self._block(key, "t", tr, tc, (nrow, self.S + 1))
        for r, job in enumerate(jobs):
            job["i64"][GE_J_POS] = bp.offset + 3 * r
            job["i64"][GE_J_T] = bt.offset + r

    # ---- user constraints (con_user.py + jac_fd.py) ---------------------
    def _g_user(self, key, fn):
        """One user group: ONE jac_fd pass of the reference over every built-in of the group.  Each built-in's rows see
        the same base state (the residue of the groups before) and depend on its own read variables only; the
        group's pass leaves one residue on every variable."""
        items = _builtins(fn)
        if not items:
            self._absent(key)
            return
        r = self._begin(key, sum(len(b.rows) for b in items))
        parts = []  # (job, srow, event index, first row of the part inside the group)
        for b in items:
            index = self.p["event_index"].get(b.event_name)
            if index is None:
                raise KeyError("unknown event %r (events: %s)" % (b.event_name, ", ".join(self.p["event_index"])))
            if isinstance(b, TableAtEvent) and not 0 <= index < self.S:
                raise ValueError("event %r starts no section: it has no first node" % b.event_name)
            srow = self.ps.index_start_u(index) + index
            k = len(b.rows)
            if isinstance(b, OrbitAtEvent):
                codes = sum(ORBIT_QUANTITIES[q] << (8 * j) for j, (q, _, _) in enumerate(b.rows))
                a = [1.0, 0.0] * 3
                for j, (_, scale, offset) in enumerate(b.rows):
                    a[2 * j], a[2 * j + 1] = scale, offset
                job = self._evt_job(GE_USER_ORBIT, -1, srow, codes, 0, r, k, 0.0, 1.0, a=a)
            else:
                job = self._tab_job(index, srow, r, b)
            parts.append((job, srow, index, r - self.group_rows[key][0]))
            r += k
        # ("dense-user", first job, its state row, every part): the first two as a group of one OrbitAtEvent has them
        self.blocks[key] = ("dense-user", parts[0][0], parts[0][1], parts)
        # jac_fd perturbs and restores EVERY variable in place (jac_fd.py:54-60)
        self._rc += 1

    def _tab_job(self, index, srow, row, fn):
        """Register a result-table job (include/gelato_b200.h: GT_*) with the residue counts of its 12 read variables."""
        reads = ([self.off["mass"] + srow] + [self.off["position"] + 3 * srow + k for k in range(3)] +
                 [self.off["velocity"] + 3 * srow + k for k in range(3)] +
                 [self.off["quaternion"] + 4 * srow + k for k in range(4)] + [self.off["t"] + index])
        lc = self.p["LaunchCondition"]
        job = {"i32": [srow, index, row, len(fn.rows), len(self._tab_rows)] + [int(self._rc[j]) for j in reads],
               "f64": [float(lc["lat"]), float(lc["lon"])], "rows": []}
        for col, scale, offset in fn.rows:
            job["rows"].append(len(self._tab_rows))
            self._tab_rows.append([TABLE_COLUMNS[col], scale, offset, -1])
        self._tab.append(job)
        return job

    # ------------------------------------------------------------------
    def _finish(self):
        self.n_rows = self._row
        self.n_coo = self._nvals
        # auxiliary tail: finite differences of the user built-ins
        for key in ("eqcon_user", "ineqcon_user"):
            b = self.blocks.get(key)
            if isinstance(b, tuple):
                for job, _, _, _ in b[3]:
                    if "rows" in job:  # result-table job: each row's values
                        for k in job["rows"]:
                            self._tab_rows[k][3] = self._nvals
                            self._nvals += AUX_PER_TABLE
                    else:
                        job["i64"][GE_J_POS] = self._nvals
                        self._nvals += AUX_PER_USER * job["i32"][GE_NROW]
        self.n_vals = self._nvals
        tmpl = np.zeros(self.n_vals, dtype=np.float64)
        for off, vals in self._tmpl:
            tmpl[off: off + vals.size] = vals
        self.vals_template = tmpl

        lin = self._lin
        self.n_lin = len(lin)
        self.lin_i32 = np.array([[r, ip, im] for r, ip, im, _, _, _ in lin], dtype=np.int32).reshape(-1, GL_I32_COLS)
        self.lin_f64 = np.array([[sp, sm, c] for _, _, _, sp, sm, c in lin], dtype=np.float64).reshape(-1, GL_F64_COLS)
        self.n_aero = len(self._aero)
        self.aero_i32 = np.array([j["i32"] for j in self._aero], dtype=np.int32).reshape(-1, GA_I32_COLS)
        self.aero_i64 = np.array([j["i64"] for j in self._aero], dtype=np.int64).reshape(-1, GA_I64_COLS)
        self.aero_f64 = np.array([j["f64"] for j in self._aero], dtype=np.float64).reshape(-1, GA_F64_COLS)
        self.n_evt = len(self._evt)
        self.evt_i32 = np.array([j["i32"] for j in self._evt], dtype=np.int32).reshape(-1, GE_I32_COLS)
        self.evt_i64 = np.array([j["i64"] for j in self._evt], dtype=np.int64).reshape(-1, GE_I64_COLS)
        self.evt_f64 = np.array([j["f64"] for j in self._evt], dtype=np.float64).reshape(-1, GE_F64_COLS)
        self.n_tab, self.n_tab_rows = len(self._tab), len(self._tab_rows)
        self.tab_i32 = np.array([j["i32"] for j in self._tab], dtype=np.int32).reshape(-1, GT_I32_COLS)
        self.tab_f64 = np.array([j["f64"] for j in self._tab], dtype=np.float64).reshape(-1, 2)
        self.tab_col = np.array([t[0] for t in self._tab_rows], dtype=np.int32)
        self.tab_sf = np.array([t[1:3] for t in self._tab_rows], dtype=np.float64).reshape(-1, 2)
        self.tab_aux = np.array([t[3] for t in self._tab_rows], dtype=np.int64)
        self.wind = np.ascontiguousarray(self.p["wind_table"], dtype=np.float64)
        self.ca = np.ascontiguousarray(self.p["ca_table"], dtype=np.float64)
        self.units = (float(self.u["mass"]), float(self.u["position"]), float(self.u["velocity"]), float(self.u["u"]),
                      float(self.u["t"]), self.dx)

    # ------------------------------------------------------------------
    # host-side views of the kernels' outputs
    def eval_counts(self):
        """Physics-leaf evaluations per objfunc and per sens call, one per
        (node x perturbation column), centre points included (SURVEY.md 8(d))."""
        n_air = n_air_fd = n_free = n_air_free = 0
        for i in range(self.S):
            n = self._sec[i][4]
            fl = int(self.sec_i32[i, GS_FLAGS])
            n_air += n if fl & GSF_AIR else 0
            n_air_fd += n if fl & GSF_AIR_FD else 0
            n_free += 0 if fl & GSF_HOLD else n
            n_air_free += n if (fl & GSF_AIR_FD) and not (fl & GSF_HOLD) else 0
        aero_rows = {0: 0, 1: 0, 2: 0}
        for j in self._aero:
            aero_rows[j["i32"][0]] += j["i32"][2]
        lanes = {GE_LLH: 5, GE_IIP: 8, GE_ANT: 5, GE_TERM: 7, GE_USER_ORBIT: 13}
        evt_jac = sum(lanes[j["i32"][0]] for j in self._evt)
        aero_jac = 13 * aero_rows[0] + 9 * aero_rows[1] + 13 * aero_rows[2]
        # result-table jobs: one output_row per job in objfunc, 18 in sens (user_table.h: lanes 0-17)
        obj = self.N + n_free + sum(aero_rows.values()) + len(self._evt) + len(self._tab)
        sens = 14 * n_air_fd + 9 * (self.N - n_air_fd) + 7 * n_free + aero_jac + evt_jac + 18 * len(self._tab)
        return {"objfunc": obj, "sens": sens, "air_nodes": n_air, "air_fd_nodes": n_air_fd,
                "noair_nodes": self.N - n_air, "free_nodes": n_free, "air_free_nodes": n_air_free,
                "aero_rows": sum(aero_rows.values()),
                "aero_jac_evals": aero_jac, "evt_jobs": len(self._evt), "evt_jac_evals": evt_jac}

    def xdep_index(self):
        """Sorted positions in `vals` of the slots that depend on x -- exactly what the
        Jacobian kernel rewrites on every call (jobs.h: dyn_scatter, aero_phase, evt_jac_phase2);
        the other slots are constants / D entries written once from `vals_template`.
        Lets a batched driver move only these values over PCIe (engine: update mode)."""
        if getattr(self, "_xdep", None) is not None:
            return self._xdep
        parts = []

        def run(start, length):
            parts.append(np.arange(start, start + length, dtype=np.int64))

        for i in range(self.S):
            n = int(self.sec_i32[i, GS_N])
            fl = int(self.sec_i32[i, GS_FLAGS])
            sj = self.sec_i64[i]
            j = np.arange(n, dtype=np.int64)
            run(sj[GS_JP_VEL], 3 * n)
            run(sj[GS_JP_T], 6 * n)
            run(sj[GS_JV_MASS], 3 * n)
            run(sj[GS_JV_POS], 9 * n)
            run(sj[GS_JV_QUAT], 12 * n)
            run(sj[GS_JV_T], 6 * n)
            if fl & GSF_AIR_FD:  # node-diagonal of the 9 dense n x (n+1) sub-blocks
                for b in range(9):
                    parts.append(sj[GS_JV_VEL] + b * n * (n + 1) + j * (n + 1) + (j + 1))
            if not fl & GSF_HOLD:
                for a in range(4):
                    for kk in range(4):
                        parts.append(sj[GS_JQ_QUAT] + (4 * j + a) * (4 * (n + 1)) + 4 * (j + 1) + kk)
                run(sj[GS_JQ_U], 8 * n)
                run(sj[GS_JQ_T], 8 * n)
        for job in self._aero:
            kind, nk = job["i32"][GA_KIND], job["i32"][GA_NK]
            run(job["i64"][GA_J_POS], 3 * nk)
            run(job["i64"][GA_J_VEL], 3 * nk)
            if kind != 1:
                run(job["i64"][GA_J_QUAT], 4 * nk)
            run(job["i64"][GA_J_T], 2 * nk)
        for job in self._evt:
            typ, nrow = job["i32"][GE_TYPE], job["i32"][GE_NROW]
            if typ == GE_TERM:
                run(job["i64"][GE_J_POS], 3 * nrow)
                run(job["i64"][GE_J_VEL], 3 * nrow)
            elif typ == GE_USER_ORBIT:
                run(job["i64"][GE_J_POS], AUX_PER_USER * nrow)
            else:
                run(job["i64"][GE_J_POS], 3)
                if typ == GE_IIP:
                    run(job["i64"][GE_J_VEL], 3)
                run(job["i64"][GE_J_T], 1)
        for aux in self.tab_aux:
            run(aux, AUX_PER_TABLE)
        idx = np.sort(np.concatenate(parts)) if parts else np.zeros(0, dtype=np.int64)
        assert idx.size == np.unique(idx).size, "an x-dependent Jacobian slot is listed twice"
        self._xdep = idx
        return idx

    @property
    def n_xdep(self):
        """Jacobian slots that depend on x (what the Jacobian kernel writes each call);
        the other n_vals - n_xdep slots are constants / D entries set once."""
        return int(self.xdep_index().size)

    def split_residuals(self, g):
        """g[n_rows] -> the reference's `funcs` dict (views into g)."""
        steps = getattr(self, "_split_steps", None)
        if steps is None:  # (key, mode, first, end) once per plan: this runs on every objfunc call
            steps = []
            for key in GROUPS:
                gr = self.group_rows.get(key)
                if gr is None:
                    steps.append((key, 0, 0, 0))
                elif key == "ineqcon_mass":  # a Python list in the reference (con_trajectory.py:61)
                    steps.append((key, 2, gr[0], gr[0] + gr[1]))
                elif key in ("eqcon_user", "ineqcon_user") and gr[1] == 1:  # one row: a scalar, like the shipped example's
                    steps.append((key, 3, gr[0], gr[0] + 1))
                else:
                    steps.append((key, 1, gr[0], gr[0] + gr[1]))
            self._split_steps = steps
        f = {"obj": g[0]}
        for key, mode, a, b in steps:
            if mode == 1:
                f[key] = g[a:b]
            elif mode == 0:
                f[key] = None
            elif mode == 2:
                f[key] = list(g[a:b])
            else:
                f[key] = g[a]
        return f

    def cost_jac(self):
        """cost_gradient.py:37-47 (constant)."""
        if self.payload_mode:
            gvec = np.zeros(self.M)
            gvec[0] = -1.0
            return {"mass": gvec}
        gvec = np.zeros(self.S + 1)
        gvec[-1] = 1.0
        return {"t": gvec}

    def _user_dense(self, vals, spec, key_order, out=None):
        """Expand the auxiliary quotients of every row of a user group into jac_fd's dense blocks
        (jac_fd.py:54-60): a variable the function does not read still gets
        (g(x after k restores) - g_base)/dx, k = how many of the variables its built-in reads were visited before it
        -- for k = 0 that is (g_base - g_base)/dx, +0 or NaN where g_base is not finite.  `out`: the dictionary of an
        earlier call to refill in place (its arrays are column slices of one (rows, n_vars) buffer, filled by one
        gather per row)."""
        order = tuple(key_order)
        nrow = sum(job["i32"][GE_NROW] if "rows" not in job else len(job["rows"]) for job, _, _, _ in spec[3])
        if out is None:
            buf = np.empty((nrow, self.n_vars))
            out, o = _UserBlocks(buf), 0
            for key in order:
                out[key] = buf[:, o: o + self.sizes[key]]
                o += self.sizes[key]
        buf = out.buffer
        for job, srow, index, r0 in spec[3]:
            if "rows" in job:
                self._table_dense(vals, job, srow, index, order, buf[r0: r0 + len(job["rows"])])
            else:
                self._orbit_dense(vals, job, srow, order, buf[r0: r0 + job["i32"][GE_NROW]])
        return out

    def _orbit_dense(self, vals, job, srow, order, buf):
        """The rows of an OrbitAtEvent job: 12 auxiliary quotients each (jobs.h: GE_USER_ORBIT)."""
        maps = self.__dict__.setdefault("_user_maps", {})
        idx = maps.get((order, srow))
        if idx is None:
            # every entry of a row is one of 13 values: q = [background quotients after 0..6 restores, the six
            # finite-difference quotients]; which one depends only on the variable's place in the perturbation order.
            # Only k = 0, 3, 6 occur (position and velocity are visited three components at a time).
            if order.index("position") > order.index("velocity"):
                raise NotImplementedError("xdict key order with velocity before position")
            parts, k = [], 0
            for key in order:
                ix = np.full(self.sizes[key], k, dtype=np.intp)
                if key in ("position", "velocity"):
                    j0 = 0 if key == "position" else 3
                    ix[3 * srow: 3 * srow + 3] = 7 + j0 + np.arange(3)
                    k += 3
                    ix[3 * srow + 3:] = k
                parts.append(ix)
            idx = maps[(order, srow)] = np.concatenate(parts)
        q = np.full(13, np.nan)  # q[1] (k = 1) is never indexed
        a0 = job["i64"][GE_J_POS]
        for r in range(buf.shape[0]):
            # background slot 0 holds k = 0 (jobs.h: evt_jac_phase1, lane 7), slots 1..5 k = 2..6
            q[0] = 0.0 * vals[a0 + 6]  # the same +0 / NaN; 0 for csr_map's probe, whose entries here stay structural zeros
            q[2:7] = vals[a0 + 7: a0 + 12]
            q[7:13] = vals[a0: a0 + 6]
            np.take(q, idx, out=buf[r])
            a0 += AUX_PER_USER

    def _table_dense(self, vals, job, srow, index, order, buf):
        """The rows of a TableAtEvent job: 18 auxiliary values each (user_table.h), taken by an index built once per
        (state row, event index, key order)."""
        maps = self.__dict__.setdefault("_user_maps", {})
        idx = maps.get((order, "table", srow, index))
        if idx is None:
            if order != tuple(VAR_ORDER):  # the device visits the read variables in the reference's key order
                raise NotImplementedError("xdict key order %s: result-table constraints follow the reference's %s"
                                          % (list(order), list(VAR_ORDER)))
            reads = {"mass": [srow], "position": [3 * srow + k for k in range(3)],
                     "velocity": [3 * srow + k for k in range(3)], "quaternion": [4 * srow + k for k in range(4)],
                     "t": [index]}
            parts, k = [], 0  # k: read variables visited so far = the next one's finite-difference slot
            for key in order:
                ix = np.empty(self.sizes[key], dtype=np.intp)
                at = 0
                for j in reads.get(key, []):
                    if j > at:
                        ix[at: j] = _TABLE_BG_SLOT[k]
                    ix[j] = k
                    k += 1
                    at = j + 1
                ix[at:] = _TABLE_BG_SLOT[k]
                parts.append(ix)
            idx = maps[(order, "table", srow, index)] = np.concatenate(parts)
        for r, row in enumerate(job["rows"]):
            a0 = self._tab_rows[row][3]
            q = np.array(vals[a0: a0 + AUX_PER_TABLE], dtype=np.float64)
            q[17] = 0.0 * q[17]  # +0 / NaN; 0 for csr_map's probe, whose entries here stay structural zeros
            np.take(q, idx, out=buf[r])

    def refresh_user_blocks(self, vals, sens_dict, key_order):
        """Refill the dense user-constraint blocks of a `funcsSens` dictionary made by split_jacobian from the SAME
        value buffer (its COO data arrays are views and already current; these blocks are computed)."""
        for key in GROUPS:
            b = self.blocks.get(key)
            if isinstance(b, tuple):
                self._user_dense(vals, b, key_order, out=sens_dict[key])

    def csr_map(self, wrt=None, key_order=VAR_ORDER):
        """The whole constraint Jacobian as ONE CSR matrix whose data is a gather of the flat value vector
        (SURVEY.md 8(f)-2): rows = the groups present, stacked in registration order
        (Trajectory_Optimization.py:358-384), columns = the variables in `key_order`; `wrt[group]`
        (optional) restricts a group to the variables it is registered against (`:358-384` wrt lists).
        Returns {"shape", "indptr", "indices", "src", "row0"}: for x-independent structure computed once,
        `data = np.append(vals, 0.0)[src]` is the CSR data of any later evaluation (`src == n_vals` marks the
        structural zeros of jac_fd's dense user blocks); entries are sorted by (row, column) and unique."""
        probe = np.arange(1, self.n_vals + 1, dtype=np.float64)  # value = slot + 1, 0.0 = constant zero
        s = self.split_jacobian(probe, key_order)
        col0, o = {}, 0
        for k in key_order:
            col0[k] = o
            o += self.sizes[k]
        rows, cols, src, row0, r0 = [], [], [], {}, 0
        for key in GROUPS:
            gr = self.group_rows.get(key)
            if gr is None:
                continue
            row0[key] = r0
            for var, blk in s[key].items():
                if wrt is not None and key in wrt and var not in wrt[key]:
                    continue
                if isinstance(blk, dict):
                    r, c, d = blk["coo"]
                else:  # dense (rows, size) block of a user constraint
                    d2 = np.atleast_2d(np.asarray(blk, dtype=np.float64))
                    r, c = np.divmod(np.arange(d2.size, dtype=np.int64), d2.shape[1])
                    d = d2.ravel()
                rows.append(np.asarray(r, dtype=np.int64) + r0)
                cols.append(np.asarray(c, dtype=np.int64) + col0[var])
                src.append(np.asarray(d, dtype=np.float64))
            r0 += gr[1]
        rows, cols, src = np.concatenate(rows), np.concatenate(cols), np.concatenate(src)
        src = np.where(src == 0.0, self.n_vals + 1, src).astype(np.int64) - 1
        order = np.lexsort((cols, rows))
        rows, cols, src = rows[order], cols[order], src[order]
        if rows.size > 1 and np.any((np.diff(rows) == 0) & (np.diff(cols) == 0)):
            raise ValueError("duplicate (row, column) entries in the constraint Jacobian")
        indptr = np.zeros(r0 + 1, dtype=np.int64)
        np.add.at(indptr, rows + 1, 1)
        return {"shape": (r0, o), "indptr": np.cumsum(indptr), "indices": cols, "src": src, "row0": row0}

    PATH_VARS = ("position", "velocity", "quaternion", "t")

    def path_rows_structure(self, layout):
        """{variable: Block} of the path rows' Jacobian (DESIGN.md section 11) from the engine's path_rows_layout():
        COO rows / cols and shape of each of position, velocity, quaternion and t, with `offset` the first of its entries
        in the row values of one scenario -- each variable one contiguous range, entries in the order the C side writes
        them (include/gelato_b200.h: gelato_plan_path_rows)."""
        acc = {var: ([], []) for var in self.PATH_VARS}
        first = {}
        for k in range(layout["n_rows"]):
            i = int(self.aero_i32[layout["job"][k], GA_SECTION])
            xa, n = self._sec[i][2], self._sec[i][4]
            off = layout["off"][k]
            for c, (var, w) in enumerate((("position", 3), ("velocity", 3), ("quaternion", 4))):
                if off[c] < 0:
                    continue
                first.setdefault(var, int(off[c]))
                cols = (w * np.arange(xa, xa + n + 1)[:, None] + np.arange(w)).ravel()
                acc[var][0].append(np.full(cols.size, k))
                acc[var][1].append(cols)
            first.setdefault("t", int(off[3]))
            acc["t"][0].append([k, k])
            acc["t"][1].append([i, i + 1])
        nr = layout["n_rows"]
        shapes = {"position": (nr, 3 * self.M), "velocity": (nr, 3 * self.M), "quaternion": (nr, 4 * self.M),
                  "t": (nr, self.S + 1)}
        out, o = {}, 0
        for var in self.PATH_VARS:
            blk = Block(o, _i4(acc[var][0]), _i4(acc[var][1]), shapes[var])
            if var in first and first[var] != o:
                raise ValueError("path-row layout is not variable-major")
            out[var] = blk
            o += blk.nnz
        if o != layout["n_vals"]:
            raise ValueError("path-row layout has %d values, the rows %d" % (layout["n_vals"], o))
        return out

    def split_jacobian(self, vals, key_order=VAR_ORDER):
        """vals[n_vals] -> the reference's `funcsSens` dict; COO data arrays are
        views into `vals` (no copies)."""
        s = {"obj": self.cost_jac()}
        for key in GROUPS:
            b = self.blocks.get(key)
            if b is None:
                s[key] = None
            elif isinstance(b, tuple):
                s[key] = self._user_dense(vals, b, key_order)
            else:
                s[key] = {var: {"coo": [blk.rows, blk.cols, vals[blk.offset: blk.offset + blk.nnz]], "shape": blk.shape}
                          for var, blk in b.items()}
        return s
