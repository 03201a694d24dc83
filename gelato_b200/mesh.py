"""Mesh accuracy of the LGR transcription (DESIGN.md section 11): the tables of the collocation error estimate, p-refinement
of the event mesh and the transfer of a solution onto the refined mesh.

    tables = mesh.grid_tables(ps)                        # once per mesh
    engine.set_mesh_grid(tables)
    err = engine.mesh_error(x)                           # [S][11] on the GPU
    events2, report = mesh.refine_nodes(events, err, tol=1e-6, n_max=30)
    ... build the problem of events2, then x2 = mesh.transfer(xdict, ps, ps2) and re-solve from x2

With GelatoProblem, `prob.path_check(xdict)` (the aero constraints between the nodes, on the same grid) can drive the
refinement too: refine_nodes(events, err, tol, n_max, path=prob.path_check(xdict)).

h-refinement: a section may be made of several LGR intervals (PSparams(..., intervals); the event keys
`mesh_intervals` / `mesh_breaks`).  Its grid has one block of test points per interval, the estimate comes per interval
(engine.mesh_error_intervals, GelatoProblem.mesh_error_intervals), and refine_nodes(..., n_min=...) splits an interval
whose degree would exceed n_max instead of capping it (the ph rule).

The estimate and the path check run on the GPU (gelato_b200.cu: k_mesh_points, k_mesh_error, k_path_points,
k_path_min); this module only builds their float64 tables once per mesh and does the host-side bookkeeping of a
refinement.
"""
import collections
import copy
import math

import numpy as np

from .problem import event_intervals
from .psparams import interval_points, lgr_diff_matrix, lgr_points


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
    tt = lgr_points(m)
    P = lagrange_basis(np.hstack((-1.0, tau)), tt)
    Q = lagrange_basis(tau, tt)
    I = np.linalg.inv(lgr_diff_matrix(m, tt)[:, 1:])
    return tt, P, Q, I


def interval_tables(tau, counts, breaks, ms):
    """(tau_t, P, Q, I) of a section made of LGR intervals (psparams.composite_tables) with ms[k] test points in interval
    k: its flipped LGR points mapped into the interval (the last one exactly its right end), P and Q rows the
    interval-local bases over its support points and its nodes (zeros elsewhere), and I block diagonal, interval k's
    block inv(lgr_diff_matrix(m_k)[:, 1:]) * w_k / 2 (the integral in section tau from the interval's start)."""
    tau = np.asarray(tau, dtype=np.float64)
    s, b, n, M = np.hstack((-1.0, tau)), np.hstack((-1.0, breaks, 1.0)), tau.size, int(sum(ms))
    tt, P, Q, I = np.empty(M), np.zeros((M, n + 1)), np.zeros((M, n)), np.zeros((M, M))
    l = c = 0
    for k, (nk, mk) in enumerate(zip(counts, ms)):
        loc = lgr_points(mk)
        tk = interval_points(loc, b[k], b[k + 1])
        tt[l:l + mk] = tk
        P[l:l + mk, c:c + nk + 1] = lagrange_basis(s[c:c + nk + 1], tk)
        Q[l:l + mk, c:c + nk] = lagrange_basis(tau[c:c + nk], tk)
        I[l:l + mk, l:l + mk] = np.linalg.inv(lgr_diff_matrix(mk, loc)[:, 1:]) * ((b[k + 1] - b[k]) / 2.0)
        l += mk
        c += nk
    return tt, P, Q, I


def grid_tables(ps, m=None):
    """The test grid of every section of `ps` (a PSparams) as gelato_plan_set_mesh_grid takes it: {"m": int32[S],
    "off": int64[S], "pool": float64[...]} with the pool laid out tau_t | P | Q | I per section.  m: None (n + 1 test
    points in a section of n nodes, n_k + 1 in each interval of n_k nodes), one count for every section (for every
    interval of a section made of several), or one per section (single-interval sections only).  When some section has
    more than one interval the grid also has {"n_int": int32[S], "int_m", "int_base": int32[sum n_int]} (test points and
    first support column of each interval)."""
    S = ps.num_sections()
    ivs = [ps.intervals(i) for i in range(S)]
    if m is None:
        mk = [[c + 1 for c in iv[0]] for iv in ivs]
    elif np.isscalar(m):
        mk = [[int(m)] * len(iv[0]) for iv in ivs]
    else:
        m = [int(v) for v in m]
        if len(m) != S or any(len(iv[0]) > 1 for iv in ivs):
            raise ValueError("a list of test-point counts needs one per section and single-interval sections, got %r"
                             % (m,))
        mk = [[v] for v in m]
    ms = [sum(v) for v in mk]
    if min(min(v) for v in mk) < 1:
        raise ValueError("one test-point count >= 1 per section is needed, got %r" % (ms,))
    parts, off, o = [], [], 0
    for i in range(S):
        if len(mk[i]) == 1:
            tt, P, Q, I = section_tables(ps.tau(i), ms[i])
        else:
            tt, P, Q, I = interval_tables(ps.tau(i), ivs[i][0], ivs[i][1], mk[i])
        off.append(o)
        for a in (tt, P, Q, I):
            parts.append(a.ravel())
            o += a.size
    out = {"m": np.array(ms, dtype=np.int32), "off": np.array(off, dtype=np.int64), "pool": np.concatenate(parts)}
    if any(len(v) > 1 for v in mk):
        out["n_int"] = np.array([len(v) for v in mk], dtype=np.int32)
        out["int_m"] = np.array([c for v in mk for c in v], dtype=np.int32)
        out["int_base"] = np.array([c for iv in ivs for c in iv[2]], dtype=np.int32)
    return out


Refinement = collections.namedtuple("Refinement", "name n_old n_new err capped path interval split",
                                    defaults=(None, 0, 1))


def _intervals(e):
    """(counts, breaks) of an event record: its `mesh_intervals` / `mesh_breaks`, else one interval."""
    iv = event_intervals(e)
    return ([int(e["num_nodes"])], np.empty(0)) if iv is None else iv


def _interval_of(b, tau):
    """The interval of breakpoints b (-1 .. +1) that holds section tau: the first k with tau <= b[k + 1] (a point on a
    breakpoint is the last node of the interval on its left)."""
    return int(np.clip(np.searchsorted(b[1:-1], tau, side="left"), 0, b.size - 2))


def _worst_path(events, path):
    """[S] (worst path residual, flight time [s] or None) per section from GelatoProblem.path_check's {(key, event
    name): (residual, time_s)} or from [S] values; +inf for a section without an aero job over it."""
    S = len(events) - 1
    if isinstance(path, dict):
        worst = {e["name"]: (np.inf, None) for e in events[:S]}
        for (_, name), (r, t) in path.items():
            if r != r or r < worst[name][0]:
                worst[name] = (r, t)
        out = [worst[e["name"]] for e in events[:S]]
    else:
        out = [(float(r), None) for r in np.asarray(path, dtype=np.float64).reshape(S)]
    r = np.array([v[0] for v in out], dtype=np.float64)
    if np.isnan(r).any() or np.isneginf(r).any():
        raise ValueError("the path residual is not finite")
    return out


def _increment(e, tol, n):
    return max(1, math.ceil(math.log(e / tol) / math.log(max(n, 2))))


def refine_nodes(events, err, tol, n_max, path=None, path_tol=1e-3, n_min=None, t_events=None):
    """ph-refinement: (new events, report).  `events` are the problem's event records (S + 1, the last one ends the
    flight), `err` the estimate: per section ([S][11], or {event name: err[11]} as GelatoProblem.mesh_error returns it)
    or per interval ([sum K][11] as engine.mesh_error_intervals returns it, or {event name: err[K][11]} as
    GelatoProblem.mesh_error_intervals does).  A section of K intervals needs K estimates.

    An interval of n nodes whose largest component error e exceeds tol wants n + P nodes, P = max(1, ceil(log(e / tol)
    / log(max(n, 2)))).  If n + P <= n_max it gets them.  Otherwise, without n_min, it gets n_max (`capped`: it stays
    above tol); with n_min it is split into B = max(2, ceil((n + P) / n_min)) equal-width intervals of n_min nodes each.
    No event is added, so time_ref chains and attitude modes keep their meaning: the new events carry `num_nodes` and,
    for a section of several intervals (or one that had the keys), `mesh_intervals` and `mesh_breaks`.  The report has
    one Refinement per interval (`interval` its index in the old section, `split` B or 1).

    path: the aero path constraints between the nodes, as GelatoProblem.path_check returns them or as [S] worst
    residuals per section.  A worst residual r below -path_tol also asks for the increment above, with -r and path_tol
    in place of e and tol, in the interval that holds the flight time of the residual (t_events: the [S + 1] event times
    in seconds of the solution the check ran on; default the records' `time`); [S] values without times apply to every
    interval of their section.  That interval's report carries r in `path` (None elsewhere and without an aero job).
    Without `path` the result is that of the estimate alone."""
    if not tol > 0.0:
        raise ValueError("tol must be positive")
    if n_min is not None and int(n_min) < 1:
        raise ValueError("n_min must be >= 1")
    S = len(events) - 1
    ivs = [_intervals(e) for e in events[:S]]
    Ks = [len(iv[0]) for iv in ivs]
    if isinstance(err, dict):
        errs = [np.asarray(err[e["name"]], dtype=np.float64).reshape(Ks[i], -1) for i, e in enumerate(events[:S])]
    else:
        a = np.asarray(err, dtype=np.float64).reshape(sum(Ks), -1)
        errs = np.split(a, np.cumsum(Ks)[:-1])
    if not all(np.isfinite(e).all() for e in errs):
        raise ValueError("the error estimate is not finite")
    if path is not None:
        if not path_tol > 0.0:
            raise ValueError("path_tol must be positive")
        path = _worst_path(events, path)
    tev = np.asarray([e["time"] for e in events] if t_events is None else t_events, dtype=np.float64)
    out = copy.deepcopy(events)
    report = []
    for i in range(S):
        counts, breaks = ivs[i]
        b = np.hstack((-1.0, breaks, 1.0))
        r, kp = None, None  # the path residual and the interval it drives (None: every interval)
        if path is not None and np.isfinite(path[i][0]):
            r, ts = float(path[i][0]), path[i][1]
            if ts is not None:
                kp = _interval_of(b, 2.0 * (ts - tev[i]) / (tev[i + 1] - tev[i]) - 1.0)
        new_counts, new_breaks = [], []
        for k, n in enumerate(counts):
            e = float(errs[i][k].max())
            want = n + _increment(e, tol, n) if e > tol else n
            rk = r if r is not None and kp in (None, k) else None
            if rk is not None and rk < -path_tol:
                want = max(want, n + _increment(-rk, path_tol, n))
            B = 1
            if want <= max(n, int(n_max)):
                n_new, capped = want, False
            elif n_min is None:
                n_new, capped = max(n, int(n_max)), True
            else:
                B = max(2, math.ceil(want / int(n_min)))
                n_new, capped = B * int(n_min), False
            if k > 0:
                new_breaks.append(float(b[k]))
            new_counts += [n_new // B] * B
            new_breaks += [float(b[k] + (b[k + 1] - b[k]) * j / B) for j in range(1, B)]
            report.append(Refinement(events[i]["name"], n, n_new, e, capped, rk, k, B))
        out[i]["num_nodes"] = int(sum(new_counts))
        if len(new_counts) > 1 or "mesh_intervals" in events[i]:
            out[i]["mesh_intervals"] = new_counts
            out[i]["mesh_breaks"] = new_breaks
    return out, report


def transfer(xdict, ps_old, ps_new):
    """A decision vector of the mesh `ps_old` moved onto `ps_new` (same sections, other node counts or intervals): the
    states at each new support point through the degree-n_k Lagrange basis over the support points of the old interval
    that holds it, the controls through the degree-(n_k - 1) basis over that interval's nodes (a point on a breakpoint
    belongs to the interval on its left, whose node it is); the event times t are unchanged.  A section whose node
    counts and breakpoints did not change is copied bit for bit."""
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
        (counts, breaks, cols), (counts2, breaks2, _) = ps_old.intervals(i), ps_new.intervals(i)
        if counts2 == counts and np.array_equal(breaks2, breaks):
            for k in width:
                X2[k][ya:yb] = X[k][xa:xb]
            U2[va:vb] = U[ua:ub]
            continue
        tau, tau2 = ps_old.tau(i), ps_new.tau(i)
        s, s2 = np.hstack((-1.0, tau)), np.hstack((-1.0, tau2))
        b = np.hstack((-1.0, breaks, 1.0))
        B, Bu = np.zeros((n2 + 1, n + 1)), np.zeros((n2, n))
        kx = np.array([_interval_of(b, t) for t in s2], dtype=int)
        for k, (nk, c) in enumerate(zip(counts, cols)):
            rx, ru = kx == k, kx[1:] == k
            B[rx, c:c + nk + 1] = lagrange_basis(s[c:c + nk + 1], s2[rx])
            Bu[ru, c:c + nk] = lagrange_basis(tau[c:c + nk], tau2[ru])
        for k in width:
            X2[k][ya:yb] = B @ X[k][xa:xb]
        U2[va:vb] = Bu @ U[ua:ub]
    out = {}
    for k in xdict:
        if k in width:
            out[k] = X2[k].ravel()
        elif k == "u":
            out[k] = U2.ravel()
        else:
            out[k] = np.array(xdict[k], dtype=np.float64, copy=True)
    return out
