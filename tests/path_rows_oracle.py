"""The path rows on the CPU oracle (TEST INFRASTRUCTURE ONLY; DESIGN.md section 11).

A numpy restatement of k_path_rows (gelato_b200/csrc/mesh_error.h: path_lane_f / path_lane_quot / path_lane_store) on
top of `oracle.nlp.OracleNLP` built with dot="seqfma", with the tables and section states of tests/mesh_oracle.py and
the evaluation of tests/path_oracle.py: the interpolation is the oracle's `o_seqfma_matmul` product, f its own
`_aero_eval`, and the finite-difference quotient the kernels' rule (tests/central_oracle.py: fd_quotient).  The row
list is the oracle's own statement of the rule.  With the gmath flavour it agrees with the kernels bit for bit.
"""
import numpy as np

from mesh_oracle import section_states, unpack


KINDS = ("alpha", "q", "qalpha")


def row_list(O, tables):
    """The path rows of the grid `tables` (include/gelato_b200.h: gelato_plan_set_path_rows), as the oracle states the
    rule: [(kind, section i, limit, test point l)] -- the aero constraints over a whole section (range "all") in aero-job
    order (alpha | q | Q-alpha, then section), each section's test points ascending, without the points whose P row is
    a unit vector (support points, where the node's own row holds the constraint)."""
    rows = []
    for kind in KINDS:
        for i, lim, rng, nk in O._aero_sections(kind):
            if rng != "all":
                continue
            n = O.ps.nodes(i)
            P = unpack(tables, i, n)[1]
            for l in range(P.shape[0]):
                if np.count_nonzero(P[l] == 1.0) == 1 and np.count_nonzero(P[l] == 0.0) == n:
                    continue
                rows.append((kind, i, lim, l))
    return rows


def path_rows(O, x, tables, mode="forward", step=None, jacobian=True):
    """(g[n_rows], vals[n_vals]) of the path rows of the decision dictionary x on the grid `tables`: g = 1 - f at each
    test point (the path check's residual there) and the Jacobian values in the layout of gelato_plan_path_rows
    (position | velocity | quaternion of kinds alpha and Q-alpha | t, each variable's rows in list order, a state row's
    entries in (node m, component c) order).  The Jacobian by the chain rule through the interpolation: per state
    component c of v_l, gq_c = -(f(v_l + dx e_c) - f(v_l)) / dx by the kernels' quotient rule, entry P[l][m] gq_c;
    per section time to / tf the same quotient with tn_l moved; mode "central": (gq(+h) + gq(-h)) * 0.5.  step: the
    step (None: the plan's dx forward, engine.DEFAULT_FD_STEP central).  jacobian=False: (g, None)."""
    from central_oracle import fd_quotient
    from gelato_b200.engine import DEFAULT_FD_STEP

    if step is None:
        step = float(O.dx) if mode == "forward" else DEFAULT_FD_STEP
    steps = [step] if mode == "forward" else [step, -step]
    units = [O.u["position"], O.u["velocity"], O.u["t"], 1.0]
    t = x["t"]
    rows = row_list(O, tables)
    g = []
    blocks = {"position": [], "velocity": [], "quaternion": [], "t": []}
    for kind, i, lim, l in rows:
        n = O.ps.nodes(i)
        tau_t, P, _, _ = unpack(tables, i, n)
        X, _ = section_states(O, x, i)
        v = O._dot(P, X)[l, 1:11]
        to, tf = t[i], t[i + 1]
        units[3] = lim

        def f(w, to_, tf_):
            w = w.reshape(1, 10)
            return O._aero_eval(kind, w[:, 0:3], w[:, 3:6], w[:, 6:10],
                                tau_t[l:l + 1] * (tf_ - to_) / 2 + (tf_ + to_) / 2, units)[0]

        f0 = f(v, to, tf)
        g.append(1.0 - f0)
        if not jacobian:
            continue

        def quot(c):
            qs = []
            for h in steps:
                w, to_, tf_ = v.copy(), to, tf
                if c < 10:
                    w[c] = w[c] + h
                elif c == 10:
                    to_ = to + h
                else:
                    tf_ = tf + h
                qs.append(-fd_quotient(f(w, to_, tf_) - f0, h))
            return qs[0] if len(qs) == 1 else (qs[0] + qs[1]) * 0.5

        gq = np.array([np.nan if (kind == "q" and 6 <= c < 10) else quot(c) for c in range(12)])
        blocks["position"].append(np.outer(P[l], gq[0:3]).ravel())
        blocks["velocity"].append(np.outer(P[l], gq[3:6]).ravel())
        if kind != "q":
            blocks["quaternion"].append(np.outer(P[l], gq[6:10]).ravel())
        blocks["t"].append(gq[10:12])
    if not jacobian:
        return np.array(g, dtype=np.float64), None
    vals = np.concatenate([np.concatenate(blocks[k]) if blocks[k] else np.zeros(0)
                           for k in ("position", "velocity", "quaternion", "t")])
    return np.array(g, dtype=np.float64), vals
