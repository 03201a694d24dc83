"""The per-interval mesh error estimate on the CPU oracle (TEST INFRASTRUCTURE ONLY; DESIGN.md section 11,
"h-refinement").

A numpy restatement of k_mesh_error on a grid whose sections may be made of LGR intervals, on top of
tests/mesh_oracle.py (the same interpolations, right-hand sides and fused multiply-add chains).  Its interval rule is
its own: it reads the intervals from the PSparams of the problem, not from the grid's interval tables.
"""
import numpy as np

from mesh_oracle import section_rhs, section_states, unpack


def mesh_error_intervals(O, x, tables):
    """(err_int[sum K][11], err[S][11]) of the decision dictionary x.  Test point l of a section belongs to the interval
    (b_k, b_k+1] of the section's breakpoints that holds tau_t[l], and is integrated from support column c_k over the
    block of I of its interval's test points.  err is the max over each section's intervals."""
    rows, err = [], np.empty((O.S, 11))
    t = x["t"]
    for i in range(O.S):
        n = O.ps.nodes(i)
        counts, breaks, cols = O.ps.intervals(i)
        b = np.hstack((-1.0, breaks, 1.0))
        tau_t, P, Q, I = unpack(tables, i, n)
        X, U = section_states(O, x, i)
        Xl, Ul = O._dot(P, X), O._dot(Q, U)
        rh = section_rhs(O, i, Xl, Ul, tau_t, t[i], t[i + 1])
        sec = []
        for k, c in enumerate(cols):
            L = np.nonzero((tau_t > b[k]) & (tau_t <= b[k + 1]))[0]
            Xh = X[c] + O._dot(I[np.ix_(L, L)], rh[L])
            sec.append(np.max(np.abs(Xh - Xl[L]), axis=0) / (1.0 + np.max(np.abs(Xl[L]), axis=0)))
        rows += sec
        err[i] = np.max(np.stack(sec), axis=0)
    return np.stack(rows), err
