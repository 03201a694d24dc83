"""Mesh accuracy of the LGR transcription (DESIGN.md section 11): the tables of the collocation error estimate, p-refinement
of the event mesh and the transfer of a solution onto the refined mesh.

    tables = mesh.grid_tables(ps)                        # once per mesh
    engine.set_mesh_grid(tables)
    err = engine.mesh_error(x)                           # [S][11] on the GPU
    events2, report = mesh.refine_nodes(events, err, tol=1e-6, n_max=30)
    ... build the problem of events2, then x2 = mesh.transfer(xdict, ps, ps2) and re-solve from x2

With GelatoProblem, `prob.path_check(xdict)` (the aero constraints between the nodes, on the same grid) can drive the
refinement too: refine_nodes(events, err, tol, n_max, path=prob.path_check(xdict)).

The estimate and the path check run on the GPU (gelato_b200.cu: k_mesh_points, k_mesh_error, k_path_points,
k_path_min); this module only builds their float64 tables once per mesh and does the host-side bookkeeping of a
refinement.
"""
import collections
import copy
import math

import numpy as np

from .psparams import lgr_diff_matrix, lgr_nodes


def lagrange_basis(support, pts):
    """B[len(pts)][len(support)]: the Lagrange basis over `support` evaluated at `pts` by the product formula.  The
    numerator and denominator of each entry are formed in the same order, so a point that equals a support point gets
    exactly 1 and 0."""
    s = np.asarray(support, dtype=np.float64)
    t = np.asarray(pts, dtype=np.float64)
    B = np.empty((t.size, s.size))
    for m in range(s.size):
        num, den = np.ones(t.size), 1.0
        for j in range(s.size):
            if j != m:
                num = num * (t - s[j])
                den = den * (s[m] - s[j])
        B[:, m] = num / den
    return B


def section_tables(tau, m):
    """(tau_t[m], P[m][n+1], Q[m][n], I[m][m]) of a section with LGR points `tau` and m test points (the flipped LGR
    points of m nodes): the state basis over {-1} U tau, the control basis over tau, and the inverse of the test grid's
    differentiation matrix without its first column (its integration matrix)."""
    tau = np.asarray(tau, dtype=np.float64)
    tt = lgr_nodes(m) if m > 1 else np.ones(1)  # one flipped LGR point: +1
    P = lagrange_basis(np.hstack((-1.0, tau)), tt)
    Q = lagrange_basis(tau, tt)
    I = np.linalg.inv(lgr_diff_matrix(m, tt)[:, 1:])
    return tt, P, Q, I


def grid_tables(ps, m=None):
    """The test grid of every section of `ps` (a PSparams) as gelato_plan_set_mesh_grid takes it: {"m": int32[S],
    "off": int64[S], "pool": float64[...]} with the pool laid out tau_t | P | Q | I per section.  m: None (n + 1 test
    points in a section of n nodes), one count for every section, or one per section."""
    S = ps.num_sections()
    if m is None:
        ms = [ps.nodes(i) + 1 for i in range(S)]
    elif np.isscalar(m):
        ms = [int(m)] * S
    else:
        ms = [int(v) for v in m]
    if len(ms) != S or min(ms) < 1:
        raise ValueError("one test-point count >= 1 per section is needed, got %r" % (ms,))
    parts, off, o = [], [], 0
    for i in range(S):
        tt, P, Q, I = section_tables(ps.tau(i), ms[i])
        off.append(o)
        for a in (tt, P, Q, I):
            parts.append(a.ravel())
            o += a.size
    return {"m": np.array(ms, dtype=np.int32), "off": np.array(off, dtype=np.int64), "pool": np.concatenate(parts)}


Refinement = collections.namedtuple("Refinement", "name n_old n_new err capped path", defaults=(None,))


def _worst_path(events, path):
    """[S] worst path residual per section from GelatoProblem.path_check's {(key, event name): (residual, time_s)} or
    from [S] values; +inf for a section without an aero job over it."""
    S = len(events) - 1
    if isinstance(path, dict):
        worst = {e["name"]: np.inf for e in events[:S]}
        for (_, name), (r, _) in path.items():
            worst[name] = r if r != r else min(worst[name], r)
        path = [worst[e["name"]] for e in events[:S]]
    path = np.asarray(path, dtype=np.float64).reshape(S)
    if np.isnan(path).any() or np.isneginf(path).any():
        raise ValueError("the path residual is not finite")
    return path


def refine_nodes(events, err, tol, n_max, path=None, path_tol=1e-3):
    """p-refinement: (new events, report).  `events` are the problem's event records (S + 1, the last one ends the
    flight), `err` the estimate per section ([S][11], or {event name: err[11]} as GelatoProblem.mesh_error returns it).

    A section whose largest component error e exceeds tol gets n + max(1, ceil(log(e / tol) / log(max(n, 2)))) nodes,
    at most n_max.  Only `num_nodes` changes: no event is added, so time_ref chains and attitude modes keep their
    meaning.  The report has one Refinement per section; `capped` marks a section that stays above tol because its
    count would exceed n_max (it is reported, not split).

    path: the aero path constraints between the nodes, as GelatoProblem.path_check returns them or as [S] worst
    residuals per section.  A section whose worst residual r is below -path_tol also gets the increment above, with -r
    and path_tol in place of e and tol; the section takes the larger of the two counts, at most n_max, and its report
    carries r in `path` (None for a section without an aero job over it).  Without `path` the result is that of the
    estimate alone."""
    if not tol > 0.0:
        raise ValueError("tol must be positive")
    S = len(events) - 1
    if isinstance(err, dict):
        err = [err[e["name"]] for e in events[:S]]
    err = np.asarray(err, dtype=np.float64).reshape(S, -1)
    if not np.isfinite(err).all():
        raise ValueError("the error estimate is not finite")
    if path is not None:
        if not path_tol > 0.0:
            raise ValueError("path_tol must be positive")
        path = _worst_path(events, path)
    out = copy.deepcopy(events)
    report = []
    for i in range(S):
        n, e = int(events[i]["num_nodes"]), float(err[i].max())
        want = n
        if e > tol:
            want = n + max(1, math.ceil(math.log(e / tol) / math.log(max(n, 2))))
        r = None
        if path is not None and np.isfinite(path[i]):
            r = float(path[i])
            if r < -path_tol:
                want = max(want, n + max(1, math.ceil(math.log(-r / path_tol) / math.log(max(n, 2)))))
        n_new = min(want, max(n, int(n_max)))
        out[i]["num_nodes"] = n_new
        report.append(Refinement(events[i]["name"], n, n_new, e, want > n_new, r))
    return out, report


def transfer(xdict, ps_old, ps_new):
    """A decision vector of the mesh `ps_old` moved onto `ps_new` (same sections, other node counts): the states of
    each section through the degree-n Lagrange basis over {-1, tau_1 .. tau_n}, the controls through the degree-(n - 1)
    basis over tau_1 .. tau_n; the event times t are unchanged.  A section whose node count did not change is copied
    bit for bit."""
    S = ps_old.num_sections()
    if ps_new.num_sections() != S:
        raise ValueError("both meshes must have the same sections")
    width = {"mass": 1, "position": 3, "velocity": 3, "quaternion": 4}
    M2, N2 = ps_new.num_x(), ps_new.num_u()
    X = {k: np.asarray(xdict[k], dtype=np.float64).reshape(-1, w) for k, w in width.items()}
    U = np.asarray(xdict["u"], dtype=np.float64).reshape(-1, 2)
    X2 = {k: np.empty((M2, w)) for k, w in width.items()}
    U2 = np.empty((N2, 2))
    for i in range(S):
        ua, ub, xa, xb, n = ps_old.get_index(i)
        va, vb, ya, yb, n2 = ps_new.get_index(i)
        if n2 == n:
            for k in width:
                X2[k][ya:yb] = X[k][xa:xb]
            U2[va:vb] = U[ua:ub]
            continue
        tau, tau2 = ps_old.tau(i), ps_new.tau(i)
        B = lagrange_basis(np.hstack((-1.0, tau)), np.hstack((-1.0, tau2)))
        for k in width:
            X2[k][ya:yb] = B @ X[k][xa:xb]
        U2[va:vb] = lagrange_basis(tau, tau2) @ U[ua:ub]
    out = {}
    for k in xdict:
        if k in width:
            out[k] = X2[k].ravel()
        elif k == "u":
            out[k] = U2.ravel()
        else:
            out[k] = np.array(xdict[k], dtype=np.float64, copy=True)
    return out
