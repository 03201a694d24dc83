"""The path check on the CPU oracle (TEST INFRASTRUCTURE ONLY; DESIGN.md section 11).

A numpy restatement of mesh_path_point / mesh_path_min (gelato_b200/csrc/mesh_error.h) on top of `oracle.nlp.OracleNLP`
built with dot="seqfma", with the tables and section states of tests/mesh_oracle.py: the interpolation is the oracle's
`o_seqfma_matmul` product and f its own `_aero_eval`, with the operations of its aero rows.  With the gmath flavour it
agrees with the kernels bit for bit.
"""
import numpy as np

from mesh_oracle import section_states, unpack


def path_check(O, x, tables):
    """(res, at), [n_aero] each in the plan's aero-job order (kind alpha | q | Q-alpha, then section): per aero job the
    smallest 1 - f over the test points of its section and the index of that test point (the first NaN if there is
    one); an "initial" job: +inf and -1.  f is the oracle's own _aero_eval, the interpolation its seqfma product and the
    time the formula of section_rhs."""
    units = [O.u["position"], O.u["velocity"], O.u["t"], 1.0]
    t = x["t"]
    res, at = [], []
    for kind in ("alpha", "q", "qalpha"):
        for i, lim, rng, nk in O._aero_sections(kind):
            if rng == "initial":
                res.append(np.inf)
                at.append(-1)
                continue
            if rng != "all":
                continue
            tau_t, P, _, _ = unpack(tables, i, O.ps.nodes(i))
            X, _ = section_states(O, x, i)
            Xl = O._dot(P, X)
            to, tf = t[i], t[i + 1]
            units[3] = lim
            r = 1.0 - O._aero_eval(kind, Xl[:, 1:4], Xl[:, 4:7], Xl[:, 7:11], tau_t * (tf - to) / 2 + (tf + to) / 2, units)
            nan = np.flatnonzero(np.isnan(r))
            k = int(nan[0]) if nan.size else int(np.argmin(r))
            res.append(r[k])
            at.append(k)
    return np.array(res, dtype=np.float64), np.array(at, dtype=np.int32)
