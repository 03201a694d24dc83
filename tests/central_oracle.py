"""Central-difference Jacobian on the CPU oracle (TEST INFRASTRUCTURE ONLY; DESIGN.md H6).

`CentralOracleNLP` is `oracle.nlp.OracleNLP` whose `sens` returns, for every Jacobian value, (s(+h) + s(-h)) * 0.5:
s(+-h) is the oracle's own forward protocol (H3, perturb/restore residue included) run with step +-h, each on its own
copy of the caller's x.  `objfunc`, sparsity and COO order are the oracle's.

The kernels form every finite-difference quotient as `num == 0 ? num : num / dx` (jobs.h: fd_div).  For dx > 0 that
is IEEE's quotient, which is what the oracle computes; for the -h pass it keeps the zero's sign where IEEE's 0 / (-h)
flips it.  The oracle divides by `self.dx`, so the passes run with `self.dx` set to a `Step`: a float that divides
by that rule and behaves as the plain number everywhere else (x += dx in place, t + dx, ...).
"""
import numpy as np

from gelato_b200.engine import fd_args
from oracle import nlp


class Step(float):
    """A finite-difference step for the oracle: `num / step` is `num` where num == 0, else IEEE's quotient."""

    def __array_ufunc__(self, ufunc, method, *inputs, **kw):
        args = tuple(float(a) if isinstance(a, Step) else a for a in inputs)
        res = getattr(ufunc, method)(*args, **kw)
        if ufunc is np.true_divide and method == "__call__" and isinstance(inputs[1], Step) and "out" not in kw:
            num = np.asarray(inputs[0], dtype=np.float64)
            res = np.where(num == 0.0, num, res)
        return res

    def __rtruediv__(self, num):
        return num if num == 0.0 else float(num) / float(self)


def fd_quotient(num, dx):
    """num / dx by the kernels' rule (what the oracle's passes compute through `Step`)."""
    return np.asarray(num, dtype=np.float64) / Step(dx)


class CentralOracleNLP(nlp.OracleNLP):
    """OracleNLP with derivative="forward" (the oracle as it is) or "central" with step fd_step (None:
    gelato_b200.engine.DEFAULT_FD_STEP); a bad mode or step raises ValueError as Engine.set_fd does."""

    def __init__(self, *args, derivative="central", fd_step=None, **kw):
        _, self.fd_step = fd_args(derivative, fd_step)
        self.derivative = derivative
        super().__init__(*args, **kw)

    def sens(self, x, funcs=None):
        if self.derivative == "forward":
            return super().sens(x, funcs)
        dx = self.dx
        try:
            self.dx = Step(self.fd_step)
            sp, _ = super().sens({k: np.array(v, dtype=np.float64, copy=True) for k, v in x.items()})
            self.dx = Step(-self.fd_step)
            sm, _ = super().sens({k: np.array(v, dtype=np.float64, copy=True) for k, v in x.items()})
        finally:
            self.dx = dx
        for grp, blk in sp.items():
            if blk is None:
                continue
            for var, b in blk.items():
                if isinstance(b, dict):
                    b["coo"][2] = (np.asarray(b["coo"][2], dtype=np.float64) +
                                   np.asarray(sm[grp][var]["coo"][2], dtype=np.float64)) * 0.5
                else:
                    blk[var] = (b + sm[grp][var]) * 0.5
        return sp, False
