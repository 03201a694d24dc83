"""A minimal stand-in for the slice of pyoptsparse the reference uses
(/root/reference/Trajectory_Optimization.py:315-416, 454-458), for machines where pyoptsparse and
IPOPT are not installed (this image): `Optimization`, `addVarGroup`, `addObj`, `addConGroup(...,
wrt=, jac=)` and a solver object called as `solver(optProb, sens=sens)`.

THE SOLVER IS NOT IPOPT.  It is scipy.optimize.minimize(method="trust-constr") (an interior-point /
trust-region SQP method) fed with the callbacks' sparse COO Jacobian blocks.  Its only purpose is an
end-to-end A/B: the same solver, the same problem, once on the CPU oracle's callbacks and once on the
CUDA callbacks -- iterates, converged payload and event times can then be compared, and the time spent
inside `objfunc` / `sens` is reported under pyoptsparse's names (`userObjTime`, `userSensTime`,
`userObjCalls`, `userSensCalls`, Trajectory_Optimization.py:511-517).  With pyoptsparse installed, use it:
the callbacks' signatures are the reference's.
"""
import time

import numpy as np
import scipy.optimize as so
import scipy.sparse as sp


class Optimization:
    def __init__(self, name, objfunc):
        self.name, self.objfunc = name, objfunc
        self.vars, self.cons, self.obj = [], [], None

    def addVarGroup(self, name, n, value=0.0, lower=None, upper=None, **_):
        self.vars.append((name, int(n), np.broadcast_to(np.asarray(value, dtype=float), (int(n),)).copy(), lower, upper))

    def addObj(self, name, **_):
        self.obj = name

    def addConGroup(self, name, n, lower=None, upper=None, wrt=None, jac=None, **_):
        self.cons.append((name, int(n), lower, upper, list(wrt) if wrt else None, jac))


class Solution:
    pass


class TrustConstr:
    """solver = TrustConstr({"maxiter": 200, "gtol": 1e-8, ...}); sol = solver(optProb, sens=sens)."""

    def __init__(self, options=None):
        self.options = dict(options or {})

    def __call__(self, prob, sens=None, **_):
        names = [v[0] for v in prob.vars]
        sizes = [v[1] for v in prob.vars]
        offs = np.concatenate(([0], np.cumsum(sizes)))
        nvar = int(offs[-1])
        col0 = dict(zip(names, offs[:-1]))
        x0 = np.concatenate([v[2] for v in prob.vars])
        lb = np.concatenate([np.full(v[1], -np.inf if v[3] is None else v[3]) for v in prob.vars])
        ub = np.concatenate([np.full(v[1], np.inf if v[4] is None else v[4]) for v in prob.vars])
        stat = {"obj_t": 0.0, "obj_n": 0, "sens_t": 0.0, "sens_n": 0}
        cache = {}

        def xdict(x):
            return {n: x[offs[i]: offs[i + 1]].copy() for i, n in enumerate(names)}

        def funcs(x):
            k = x.tobytes()
            if cache.get("fk") != k:
                t0 = time.perf_counter()
                f, fail = prob.objfunc(xdict(x))
                stat["obj_t"] += time.perf_counter() - t0
                stat["obj_n"] += 1
                assert not fail
                cache["fk"], cache["f"] = k, f
            return cache["f"]

        def jacs(x):
            k = x.tobytes()
            if cache.get("jk") != k:
                f = funcs(x)
                t0 = time.perf_counter()
                s, fail = sens(xdict(x), f)
                stat["sens_t"] += time.perf_counter() - t0
                stat["sens_n"] += 1
                assert not fail
                cache["jk"], cache["j"] = k, s
            return cache["j"]

        def con_vec(groups):
            def f(x):
                fx = funcs(x)
                return np.concatenate([np.atleast_1d(np.asarray(fx[g[0]], dtype=float)) for g in groups])
            return f

        def con_jac(groups):
            nrow = sum(g[1] for g in groups)

            def j(x):
                s = jacs(x)
                rows, cols, data = [], [], []
                r0 = 0
                for name, n, _, _, wrt, _ in groups:
                    for var, blk in s[name].items():
                        if wrt is not None and var not in wrt:
                            continue
                        if isinstance(blk, dict):
                            r, c, d = blk["coo"]
                        else:
                            dense = sp.coo_matrix(np.atleast_2d(np.asarray(blk, dtype=float)))
                            r, c, d = dense.row, dense.col, dense.data
                        rows.append(np.asarray(r) + r0)
                        cols.append(np.asarray(c) + col0[var])
                        data.append(np.asarray(d, dtype=float))
                    r0 += n
                return sp.coo_matrix((np.concatenate(data), (np.concatenate(rows), np.concatenate(cols))),
                                     shape=(nrow, nvar)).tocsr()
            return j

        eq = [g for g in prob.cons if g[3] is not None and g[2] == g[3]]
        ineq = [g for g in prob.cons if g not in eq]
        constraints = []
        if eq:
            v = np.concatenate([np.full(g[1], g[2]) for g in eq])
            constraints.append(so.NonlinearConstraint(con_vec(eq), v, v, jac=con_jac(eq), hess=so.BFGS()))
        if ineq:
            lo = np.concatenate([np.full(g[1], -np.inf if g[2] is None else g[2]) for g in ineq])
            hi = np.concatenate([np.full(g[1], np.inf if g[3] is None else g[3]) for g in ineq])
            constraints.append(so.NonlinearConstraint(con_vec(ineq), lo, hi, jac=con_jac(ineq), hess=so.BFGS()))

        def obj(x):
            return float(funcs(x)[prob.obj])

        def grad(x):
            g = np.zeros(nvar)
            for var, blk in jacs(x)[prob.obj].items():
                g[col0[var]: col0[var] + np.size(blk)] = np.ravel(blk)
            return g

        opts = {"maxiter": 300, "gtol": 1e-8, "xtol": 1e-10, "verbose": 0, "sparse_jacobian": True}
        opts.update(self.options)
        history = []
        t0 = time.perf_counter()
        res = so.minimize(obj, x0, jac=grad, hess=so.BFGS(), method="trust-constr", bounds=so.Bounds(lb, ub, keep_feasible=False),
                          constraints=constraints, options=opts,
                          callback=lambda xk, st: history.append((st.fun, st.constr_violation)) and False)
        sol = Solution()
        sol.xStar = xdict(res.x)
        sol.fStar = res.fun
        sol.optTime = time.perf_counter() - t0
        sol.userObjTime, sol.userObjCalls = stat["obj_t"], stat["obj_n"]
        sol.userSensTime, sol.userSensCalls = stat["sens_t"], stat["sens_n"]
        sol.constr_violation = float(res.constr_violation)
        sol.nit, sol.status, sol.message, sol.history = int(res.nit), int(res.status), str(res.message), history
        return sol


# registration of the reference's variable groups, bounds and constraint groups
VAR_BOUNDS = {"mass": (1.0e-9, 2.0), "position": (-10.0, 10.0), "velocity": (-20.0, 20.0), "quaternion": (-1.0, 1.0),
              "u": (-9.0, 9.0), "t": (0.0, 1.5)}
WRT = {
    "eqcon_init": ["mass", "position", "velocity", "quaternion"], "eqcon_time": ["t"], "eqcon_dyn_mass": ["mass", "t"],
    "eqcon_dyn_pos": ["position", "velocity", "t"], "eqcon_dyn_vel": ["mass", "position", "velocity", "quaternion", "t"],
    "eqcon_dyn_quat": ["quaternion", "u", "t"], "eqcon_knot": ["mass", "position", "velocity", "quaternion"],
    "eqcon_terminal": ["position", "velocity"], "eqcon_rate": ["u"], "eqcon_pos": ["position", "t"],
    "eqcon_iip": ["position", "velocity", "t"], "eqcon_user": ["mass", "position", "velocity", "quaternion", "u", "t"],
    "ineqcon_alpha": ["position", "velocity", "quaternion", "t"], "ineqcon_q": ["position", "velocity", "quaternion", "t"],
    "ineqcon_qalpha": ["position", "velocity", "quaternion", "t"], "ineqcon_mass": ["mass"], "ineqcon_kick": ["u"],
    "ineqcon_time": ["t"], "ineqcon_pos": ["position", "t"], "ineqcon_iip": ["position", "velocity", "t"],
    "ineqcon_antenna": ["position", "t"], "ineqcon_user": ["mass", "position", "velocity", "quaternion", "u", "t"],
    # the aero constraints between the nodes (GelatoProblem(..., path_grid=...); DESIGN.md section 11)
    "ineqcon_path": ["position", "velocity", "quaternion", "t"],
}


def register(objfunc, sens, xdict_init, condition, Opt=Optimization):
    """The registration block of the reference driver (Trajectory_Optimization.py:315-416), for any
    pyoptsparse-compatible `Opt` class."""
    prob = Opt("Rocket trajectory optimization", objfunc)
    for name in ("mass", "position", "velocity", "quaternion", "u", "t"):
        lo, hi = VAR_BOUNDS[name]
        prob.addVarGroup(name, len(xdict_init[name]), value=xdict_init[name], lower=lo, upper=hi)
    f_init = objfunc(xdict_init)[0]
    jac_init = sens(xdict_init, f_init)[0]
    wrt = dict(WRT)
    if condition["OptimizationMode"] == "Payload":
        wrt["eqcon_init"] = ["position", "velocity", "quaternion"]
    for key, val in f_init.items():
        if key == "obj":
            prob.addObj("obj")
        elif val is not None:
            n = len(val) if hasattr(val, "__len__") else 1
            prob.addConGroup(key, n, lower=0.0, upper=None if "ineqcon" in key else 0.0, wrt=wrt[key], jac=jac_init[key])
    return prob


def attach_structure(prob, pdict):
    """Tell a solver of this package where the non-linear couplings of the transcription are (ipsolve.py's sparse
    finite-difference Hessian): sizes and, per section, (first control row, first state row, nodes).  pyoptsparse has
    no use for it; the attribute is ignored by anything else."""
    ps = pdict["ps_params"]
    S = int(pdict["num_sections"])
    prob.structure = {"M": int(pdict["M"]), "N": int(pdict["N"]), "S": S,
                      "sections": [(ps.get_index(i)[0], ps.get_index(i)[2], ps.get_index(i)[4]) for i in range(S)]}
    return prob
