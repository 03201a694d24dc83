"""Drop-in for the hot-path part of the reference's `lib` package.

The reference's callbacks are assembled from per-group functions with the
signature `f(xdict, pdict, unitdict, condition)` in lib/con_dynamics.py,
con_aero.py, con_waypoint.py, con_init_terminal_knot.py, con_trajectory.py,
con_user.py, plus cost_gradient.py and jac_fd.py
(/root/reference/Trajectory_Optimization.py:194-312).  The modules of this
package keep those names and signatures, so code (or tests) written against
individual groups keeps working:

    from gelato_b200.lib import con_dynamics
    r = con_dynamics.equality_dynamics_velocity(xdict, pdict, unitdict, condition)
    J = con_dynamics.equality_jac_dynamics_velocity(xdict, pdict, unitdict, condition)

Behind them sits ONE GelatoProblem per `pdict` (compiled on first use) and a
one-entry cache per callback kind keyed on the decision vector: the 23 value
functions of an `objfunc` cost one residual-kernel launch, the 23 Jacobian
functions of a `sens` one Jacobian-kernel launch.

Semantics note.  A Jacobian group returns the values it has INSIDE the
reference's `sens` call sequence (Trajectory_Optimization.py:247-309): groups
evaluated earlier leave a rounding residue `fl(fl(x+dx)-dx)` in `xdict`, which
later groups' finite differences see (DESIGN.md "H3").  Calling a reference
group function on a pristine `xdict` differs from that by finite-difference
noise only.  The caller's `xdict` is never modified here.
"""
import numpy as np

from .. import callbacks as _cb
from ..plan import VAR_ORDER

_config = {"user_eq": None, "user_ineq": None, "device": 0, "coord": None, "engine_factory": None}
_problems = {}  # id(pdict) -> _Cached


def configure(user_eq=None, user_ineq=None, device=0, coord=None, engine_factory=None):
    """Built-in user constraints (e.g. PerigeeAtEvent("IIP_END"), TableAtEvent("FAIRING", [("altitude", 1e5, 1.0)]), or
    a list of them) and the CUDA device used
    by problems created from now on.  Arbitrary Python user constraints stay on the host:
    evaluate them with the reference's own con_user / jac_fd (jac_fd below accepts them)."""
    _config.update(user_eq=user_eq, user_ineq=user_ineq, device=device, coord=coord, engine_factory=engine_factory)
    reset()


def reset():
    """Drop every cached problem (frees their GPU plans)."""
    for c in _problems.values():
        c.prob.close()
    _problems.clear()


class _Cached:
    def __init__(self, pdict, unitdict, condition):
        self.pdict = pdict  # keeps id(pdict) alive
        self.prob = _cb.GelatoProblem(pdict, unitdict, condition, user_eq=_config["user_eq"],
                                      user_ineq=_config["user_ineq"], device=_config["device"],
                                      coord=_config["coord"], engine_factory=_config["engine_factory"])
        self._fx = self._jx = None
        self._f = self._j = None

    def _key(self, xdict):
        return self.prob.pack(xdict).tobytes()

    def funcs(self, xdict):
        k = self._key(xdict)
        if k != self._fx:
            self._f, self._fx = self.prob.objfunc(xdict)[0], k
        return self._f

    def sens(self, xdict):
        k = self._key(xdict) + repr([n for n in xdict if n in VAR_ORDER]).encode()
        if k != self._jx:
            self._j, self._jx = self.prob.sens(xdict)[0], k
        return self._j


def problem_for(pdict, unitdict, condition):
    c = _problems.get(id(pdict))
    if c is None or c.pdict is not pdict:
        c = _problems[id(pdict)] = _Cached(pdict, unitdict, condition)
    return c


def _value(key):
    def f(xdict, pdict, unitdict, condition):
        v = problem_for(pdict, unitdict, condition).funcs(xdict)[key]
        return None if v is None else (list(v) if isinstance(v, list) else np.array(v, copy=True))

    f.__doc__ = "funcs[%r] of the reference's objfunc, evaluated by the residual kernel." % key
    return f


def _jacobian(key):
    def f(xdict, pdict, unitdict, condition):
        blk = problem_for(pdict, unitdict, condition).sens(xdict)[key]
        if blk is None:
            return None
        out = {}
        for var, b in blk.items():
            if isinstance(b, dict):
                out[var] = {"coo": [b["coo"][0], b["coo"][1], np.array(b["coo"][2], copy=True)], "shape": b["shape"]}
            else:
                out[var] = np.array(b, copy=True)
        return out

    f.__doc__ = "funcsSens[%r] of the reference's sens, evaluated by the Jacobian kernel." % key
    return f


def _length(key):
    def f(xdict, pdict, unitdict, condition):
        gr = problem_for(pdict, unitdict, condition).prob.plan.group_rows.get(key)
        return 0 if gr is None else int(gr[1])

    f.__doc__ = "Row count of funcs[%r]." % key
    return f
