"""Drop-in `objfunc` / `sens` callbacks backed by the CUDA engine.

Same signatures and return structures as the reference's callbacks
(/root/reference/Trajectory_Optimization.py:194-242 `objfunc(xdict) -> (funcs,
fail)`, :245-312 `sens(xdict, funcs) -> (funcsSens, fail)`), so pyoptsparse /
IPOPT consume them unchanged:

    prob = GelatoProblem(pdict, unitdict, condition, user_eq=PerigeeAtEvent("IIP_END"))
    optProb = Optimization("Rocket trajectory optimization", prob.objfunc)
    ... addVarGroup / addConGroup(jac=prob.sens(x0, prob.objfunc(x0)[0])[0][key]) ...
    IPOPT(options)(optProb, sens=prob.sens)

One call = one host->device copy of x, ONE kernel launch, one device->host copy
of the whole result, sliced into the reference's dictionaries as views.
`fail` is always False, like the reference (:240,311); CUDA errors raise.
"""
import numpy as np

from . import engine as _engine
from .plan import (GROUPS, ORBIT_QUANTITIES, TABLE_COLUMNS, VAR_ORDER, CompiledPlan, OrbitAtEvent,  # noqa: F401
                   PerigeeAtEvent, TableAtEvent)


class GelatoProblem:
    def __init__(self, pdict, unitdict, condition, user_eq=None, user_ineq=None, device=0, coord=None,
                 engine_factory=None, reuse_output=True, fuse_pair=False, derivative="forward", fd_step=None,
                 path_grid=None):
        """engine_factory(plan) -> object with eval_residuals / eval_jacobian / close / launches;
        default: the CUDA engine on `device` (the CPU test tier passes the host emulator of the
        kernels, tests/emu_binding.py, to exercise this host logic without a GPU).

        reuse_output=True (default): `sens` writes into ONE page-locked buffer kept across calls and only the
        x-dependent Jacobian values cross PCIe (update mode); the returned COO data arrays are views of that
        buffer, valid until the next `sens` call -- what pyoptsparse needs (it converts them at once), and ~10x
        less traffic on fine meshes.  reuse_output=False: fresh arrays on every call, like the reference.

        fuse_pair=True (needs reuse_output): every `objfunc` call runs the PAIR evaluation -- the Jacobian launch
        that also writes objfunc's rows -- and keeps the Jacobian; a `sens` call at the same decision vector (what a
        solver does after it accepts a point) then returns it without touching the GPU.  Same values bit for bit;
        one call of ~0.07 ms instead of two for the shipped example, at the price of a Jacobian download for every
        objfunc call that no sens follows (line-search trial points).

        derivative="forward" (default): the reference's forward-difference Jacobian, bit for bit.  "central": central
        differences with step fd_step (None: engine.DEFAULT_FD_STEP) -- 100-1000x closer to the derivative on most
        blocks for about twice the Jacobian's GPU time; same sparsity, same objfunc (DESIGN.md H6).  `sens`,
        `jacobian_csr` and the fused pair follow it; `engine.set_fd` switches it later.

        path_grid=None (default): the NLP as the reference has it.  A test grid ({"m", "off", "pool"} as
        gelato_b200.mesh.grid_tables builds it, e.g. mesh.grid_tables(plan.ps) for n + 1 points per section): the aero
        constraints are also enforced between the nodes, as the inequality group "ineqcon_path" -- one row per test point
        of every aero constraint over a whole section, except the points that are nodes (DESIGN.md section 11).
        `objfunc`, `sens` and `jacobian_csr` add the group after the others; every other key is unchanged bit for bit.
        path_rows_index() names the rows."""
        _engine.fd_args(derivative, fd_step)  # a bad mode or step fails before anything is built
        self.plan = CompiledPlan(pdict, unitdict, condition, user_eq=user_eq, user_ineq=user_ineq, coord=coord)
        self.engine = engine_factory(self.plan) if engine_factory else _engine.Engine(self.plan, device=device)
        if derivative != "forward":
            self.engine.set_fd(derivative, fd_step)
        self.reuse_output = bool(reuse_output) and hasattr(self.engine, "eval_jacobian_update")
        self._vals = None
        self._csr = None
        self._x = np.empty(self.plan.n_vars)
        self._sizes = [self.plan.sizes[k] for k in VAR_ORDER]
        self._sens_dict = None
        self.fuse_pair = bool(fuse_pair) and self.reuse_output and hasattr(self.engine, "eval_pair_update")
        self._x_pair = None  # the decision vector the kept Jacobian belongs to
        self._pair_fresh = False
        self._mesh_grid = None  # the tables of the engine's mesh grid (mesh.grid_tables), once set
        # path rows: their layout (engine.path_rows_layout) and COO blocks (plan.path_rows_structure), and the Jacobian
        # buffer funcsSens["ineqcon_path"] views (reuse_output; the fused pair fills it from objfunc)
        self._path = self._path_vals = None
        if path_grid is not None:
            self.engine.set_path_rows(path_grid)
            layout = self.engine.path_rows_layout()
            self._path = (layout, self.plan.path_rows_structure(layout))

    # -- helpers ---------------------------------------------------------
    def pack(self, xdict):
        """xdict -> flat decision vector in the engine's order (mass | position |
        velocity | quaternion | u | t), independent of the dict's key order."""
        try:  # the usual case -- six 1-D arrays of the right sizes -- in one C call
            parts = [xdict[k] for k in VAR_ORDER]
            if [len(v) for v in parts] == self._sizes:
                np.concatenate(parts, out=self._x)
                return self._x
        except (ValueError, TypeError):
            pass
        o = 0
        for k in VAR_ORDER:
            n = self.plan.sizes[k]
            v = np.asarray(xdict[k], dtype=np.float64).ravel()
            if v.size != n:
                raise ValueError("xdict[%r] has %d entries, expected %d" % (k, v.size, n))
            self._x[o: o + n] = v
            o += n
        return self._x

    # -- the two callbacks -------------------------------------------------
    def _output_buffer(self):
        if self._vals is None:
            alloc = getattr(self.engine, "alloc_output", None)  # the CUDA engine: page-locked memory
            self._vals = alloc(self.plan.n_vals) if alloc else _engine.PinnedArray(self.plan.n_vals)
            self.engine.jacobian_template(self._vals.array, 1)
        return self._vals.array

    def objfunc(self, xdict):
        x = self.pack(xdict)
        if self.fuse_pair:
            g = np.empty(self.plan.n_rows)
            self.engine.eval_pair_update(x, g, self._output_buffer(), 1)
            if self._x_pair is None:
                self._x_pair = np.empty_like(x)
            self._x_pair[:] = x
            self._pair_fresh = True
            return self._with_path(self.plan.split_residuals(g), x, self._path_buffer()), False
        g = self.engine.eval_residuals(x)
        return self._with_path(self.plan.split_residuals(g), x, None), False

    def _with_path(self, funcs, x, vals):
        """funcs plus "ineqcon_path" (with path rows); vals: a buffer for the rows' Jacobian at x, or None."""
        if self._path is not None:
            funcs["ineqcon_path"] = self.engine.eval_path_rows(x, out=(np.empty(self._path[0]["n_rows"]), vals))[0]
        return funcs

    def _path_buffer(self):
        """The one buffer of the path rows' Jacobian values kept across calls (reuse_output)."""
        if self._path_vals is None and self._path is not None:
            alloc = getattr(self.engine, "alloc_output", None)  # the CUDA engine: page-locked memory
            self._path_vals = alloc(self._path[0]["n_vals"]) if alloc else _engine.PinnedArray(self._path[0]["n_vals"])
        return None if self._path_vals is None else self._path_vals.array

    def _path_sens(self, vals):
        """funcsSens["ineqcon_path"]: the COO blocks with data arrays that are views of vals."""
        return {var: {"coo": [b.rows, b.cols, vals[b.offset: b.offset + b.nnz]], "shape": b.shape}
                for var, b in self._path[1].items()}

    def _path_jacobian(self, x):
        """The path rows' Jacobian values at x in a fresh array."""
        return self.engine.eval_path_rows(x, out=(None, np.empty(self._path[0]["n_vals"])))[1]

    def sens(self, xdict, funcs=None):
        if self.reuse_output:
            x = self.pack(xdict)
            if self.fuse_pair and self._x_pair is not None and self._pair_fresh and np.array_equal(x, self._x_pair):
                vals = self._output_buffer()  # already holds this point's Jacobian (and the path rows')
            else:
                vals = self.engine.eval_jacobian_update(x, self._output_buffer(), 1)
                self._pair_fresh = False
                if self._path is not None:
                    self.engine.eval_path_rows(x, out=(None, self._path_buffer()))
            # the dictionary is built once per key order: its COO data arrays are views of the one buffer the engine
            # refreshes in place; only the dense user-constraint blocks are recomputed
            order = tuple(k for k in xdict.keys() if k in VAR_ORDER)
            if self._sens_dict is None or self._sens_dict[0] != order or self._sens_dict[2] is not vals:
                self._sens_dict = (order, self.plan.split_jacobian(vals, key_order=list(order)), vals)
                if self._path is not None:
                    self._sens_dict[1]["ineqcon_path"] = self._path_sens(self._path_buffer())
            else:
                self.plan.refresh_user_blocks(vals, self._sens_dict[1], order)
            return self._sens_dict[1], False
        x = self.pack(xdict)
        vals = self.engine.eval_jacobian(x)
        s = self.plan.split_jacobian(vals, key_order=[k for k in xdict.keys() if k in VAR_ORDER])
        if self._path is not None:
            s["ineqcon_path"] = self._path_sens(self._path_jacobian(x))
        return s, False

    def jacobian_csr(self, xdict, wrt=None):
        """The constraint Jacobian of all registered groups as one scipy CSR matrix (rows in registration order,
        columns in `xdict` key order): the structure is compiled once (`plan.csr_map`), each call is one kernel
        launch and one gather -- no per-call COO sorting (what pyoptsparse does with the dictionaries of `sens`).
        `wrt`: {group: [variables]} as in Trajectory_Optimization.py:358-384 (None = every block).  With path rows,
        "ineqcon_path" comes last."""
        import scipy.sparse as sp

        order = tuple(k for k in xdict.keys() if k in VAR_ORDER)
        key = (order, None if wrt is None else tuple(sorted((g, tuple(v)) for g, v in wrt.items())))
        if self._csr is None or self._csr[0] != key:
            self._csr = (key, self.plan.csr_map(wrt=wrt, key_order=order))
        m = self._csr[1]
        x = self.pack(xdict)
        vals = self.engine.eval_jacobian(x)
        data = np.append(vals, 0.0)[m["src"]]
        J = sp.csr_matrix((data, m["indices"], m["indptr"]), shape=m["shape"])
        if self._path is None:
            return J
        pv = self._path_jacobian(x)
        col0 = dict(zip(order, np.cumsum([0] + [self.plan.sizes[k] for k in order])))
        rows, cols, data = [], [], []
        for var, b in self._path[1].items():
            if wrt is not None and "ineqcon_path" in wrt and var not in wrt["ineqcon_path"]:
                continue
            rows.append(b.rows)
            cols.append(b.cols.astype(np.int64) + col0[var])
            data.append(pv[b.offset: b.offset + b.nnz])
        Jp = sp.csr_matrix((np.concatenate(data), (np.concatenate(rows), np.concatenate(cols))),
                           shape=(self._path[0]["n_rows"], J.shape[1]))
        return sp.vstack([J, Jp], format="csr")

    def path_rows_index(self):
        """[(funcs key of the aero constraint, event name, test point l)] of the rows of funcs["ineqcon_path"], in
        order (the test point is tau_t[l] of the path grid's section); [] without path rows."""
        if self._path is None:
            return []
        lay = self._path[0]
        return [(self._AERO_KEYS[self.plan.aero_i32[j, 0]], self.plan.p["params"][self.plan.aero_i32[j, 1]]["name"], int(l))
                for j, l in zip(lay["job"], lay["l"])]

    def mesh_error(self, xdict):
        """{event name: err[11]}: the collocation error estimate of each section between its nodes, per state component
        (mass | position 3 | velocity 3 | quaternion 4), on the default test grid (n + 1 points, set on first use).
        gelato_b200.mesh.refine_nodes takes the result as it is (DESIGN.md section 11)."""
        self._default_mesh_grid()
        err = self.engine.mesh_error(self.pack(xdict))
        return {prm["name"]: err[i] for i, prm in enumerate(self.plan.p["params"][: self.plan.S])}

    def mesh_error_intervals(self, xdict):
        """{event name: err[K][11]}: mesh_error per LGR interval of each section (K = 1 for a section of one interval;
        a section's row of mesh_error is the max over its intervals).  refine_nodes takes it as it is."""
        self._default_mesh_grid()
        err = self.engine.mesh_error_intervals(self.pack(xdict))
        out, k = {}, 0
        for i, prm in enumerate(self.plan.p["params"][: self.plan.S]):
            K = len(self.plan.ps.intervals(i)[0])
            out[prm["name"]] = err[k:k + K]
            k += K
        return out

    _AERO_KEYS = ("ineqcon_alpha", "ineqcon_q", "ineqcon_qalpha")

    def path_check(self, xdict):
        """{(funcs key, event name): (residual, time_s)}: for each aero constraint over a whole section (range "all"),
        the smallest value of its row's expression 1 - f / limit between the nodes -- on the default test grid (n + 1
        points, set on first use and shared with mesh_error) -- and the flight time [s] of the test point where it
        occurs.  The NLP only holds the rows at the nodes; a negative residual is a violation in between.
        gelato_b200.mesh.refine_nodes takes the result as its `path` argument (DESIGN.md section 11)."""
        tables = self._default_mesh_grid()
        x = self.pack(xdict)
        res, at = self.engine.path_check(x)
        t = x[-(self.plan.S + 1):]
        out = {}
        for j, (kind, i, nk, _) in enumerate(self.plan.aero_i32):
            if nk == 1:  # "initial": a point constraint, nothing between nodes
                continue
            to, tf = t[i], t[i + 1]
            tau = tables["pool"][tables["off"][i] + at[j]]  # tau_t[at] of section i
            out[(self._AERO_KEYS[kind], self.plan.p["params"][i]["name"])] = (
                float(res[j]), float((tau * (tf - to) / 2 + (tf + to) / 2) * self.plan.units[4]))
        return out

    def _default_mesh_grid(self):
        """The grid of mesh_error and path_check (n + 1 test points per section): set on the engine on first use."""
        if self._mesh_grid is None:
            from . import mesh

            tables = mesh.grid_tables(self.plan.ps)
            self.engine.set_mesh_grid(tables)
            self._mesh_grid = tables
        return self._mesh_grid

    # -- flat-vector variants (no dictionaries), used by benchmarks / batched drivers
    def residuals(self, x, n_scen=1):
        return self.engine.eval_residuals(x, n_scen)

    def jacobian_values(self, x, n_scen=1):
        return self.engine.eval_jacobian(x, n_scen)

    def close(self):
        for buf in (self._vals, self._path_vals):
            if buf is not None:
                buf.free()
        self._vals = self._path_vals = None
        self.engine.close()


def make_callbacks(pdict, unitdict, condition, user_eq=None, user_ineq=None, device=0):
    """(objfunc, sens) closures with the reference's signatures."""
    prob = GelatoProblem(pdict, unitdict, condition, user_eq=user_eq, user_ineq=user_ineq, device=device)
    return prob.objfunc, prob.sens
