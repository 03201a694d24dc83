"""Path rows: the aero constraints as NLP rows at the test points between the nodes (DESIGN.md section 11).

CPU tier: the kernels' code in the host emulator against tests/path_rows_oracle.py bit for bit (variants, both modes, two
grids, three decision vectors), the row list and its counts, the rows against the path check, the derivative against
4th-order differences, GelatoProblem with and without `path_grid`, refusals and the edge-state catalogue.
GPU tier: the C ABI against the oracle bit for bit (variants, a dispersed batch with per-scenario blocks, the benchmark
workload), host / pinned / device entry points, and residual-only calls."""
import ctypes

import numpy as np
import pytest

import emu_path_rows
import helpers
import mesh_oracle
import path_rows_oracle
import test_edge_states as edge
from gelato_b200 import callbacks, engine, mesh, nlpshim, problem, scenarios
from gelato_b200.plan import GROUPS
from oracle import leaves

VARIANTS = [("example", 1), ("all_aero", 1), ("three_stage", 1), ("neg_area", 1), ("example", 15)]
MODES = ("forward", "central")
AERO_KEYS = ("ineqcon_alpha", "ineqcon_q", "ineqcon_qalpha")


def _bits(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64)).view(np.int64)


def _eq(a, b):
    return np.shape(a) == np.shape(b) and np.array_equal(_bits(a), _bits(b))


_CACHE = {}


def _setup(variant, factor=1):
    if (variant, factor) not in _CACHE:
        Lg = leaves.get("gmath")
        p, u, c, x0 = problem.problem_from_inputs(helpers.variant_inputs(variant), coord=Lg.coordinate_c, factor=factor,
                                                  max_nodes=20)
        O = helpers.oracle_nlp(p, u, c, "gmath", "seqfma")
        _CACHE[(variant, factor)] = (p, u, c, x0, O, helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c))
    return _CACHE[(variant, factor)]


def _solution(P):
    x = np.load(helpers.GOLDEN + "/example_solution.npz")["x"]
    return problem.vector_to_xdict(x, P.M, P.N, P.S)


def _points(x0, P, variant, factor):
    return [x0, helpers.perturbed(x0)] + ([_solution(P)] if (variant, factor) == ("example", 1) else [])


def _grids(ps):
    """The default grid (n + 1 points) and m = 2n + 1."""
    return [mesh.grid_tables(ps), mesh.grid_tables(ps, m=[2 * ps.nodes(i) + 1 for i in range(ps.num_sections())])]


def _want_layout(O, P, tabs):
    """(job, l) of every row by the oracle's statement of the rule, jobs numbered in the plan's aero-job order."""
    jobs = {(int(k), int(i)): j for j, (k, i, nk, _) in enumerate(P.aero_i32)}
    return [(jobs[(path_rows_oracle.KINDS.index(kind), i)], l) for kind, i, _, l in path_rows_oracle.row_list(O, tabs)]


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("variant,factor", VARIANTS)
def test_emulator_equals_oracle_bit_for_bit(variant, factor):
    p, u, c, x0, O, P = _setup(variant, factor)
    E = emu_path_rows.PathRowsEmuEngine(P)
    for tabs in _grids(O.ps):
        E.set_path_rows(tabs)
        lay = E.path_rows_layout()
        assert list(zip(lay["job"], lay["l"])) == _want_layout(O, P, tabs)
        for mode in MODES:
            E.set_fd(mode)
            for x in _points(x0, P, variant, factor):
                g, v = E.eval_path_rows(problem.xdict_to_vector(x))
                gw, vw = path_rows_oracle.path_rows(O, x, tabs, mode)
                assert g.shape == (lay["n_rows"],) and v.shape == (lay["n_vals"],)
                assert _eq(g, gw) and _eq(v, vw), mode


def test_row_counts_and_the_support_point_rule():
    counts = {("example", 1): (1, 16, 2752), ("all_aero", 1): (3, 37, 5694), ("example", 15): (12, 240, 50880)}
    for (variant, factor), (jobs, rows, vals) in counts.items():
        p, u, c, x0, O, P = _setup(variant, factor)
        E = emu_path_rows.PathRowsEmuEngine(P)
        E.set_path_rows(mesh.grid_tables(O.ps))
        lay = E.path_rows_layout()
        assert (len(set(lay["job"])), lay["n_rows"], lay["n_vals"]) == (jobs, rows, vals), variant
        assert not (P.aero_i32[lay["job"], 2] == 1).any()  # "initial" jobs have no rows
    # a grid whose interior test point 3 of every section of 4+ nodes is moved onto LGR node 2: that point is dropped too
    p, u, c, x0, O, P = _setup("all_aero")
    tabs = mesh.grid_tables(O.ps)
    pool = tabs["pool"].copy()
    moved = [i for i in range(O.S) if O.ps.nodes(i) >= 4]
    for i in moved:
        n, o = O.ps.nodes(i), int(tabs["off"][i])
        M = int(tabs["m"][i])
        pool[o + 3] = O.ps.tau(i)[2]
        pool[o + M + 3 * (n + 1): o + M + 4 * (n + 1)] = mesh.lagrange_basis(np.hstack((-1.0, O.ps.tau(i))), pool[o + 3:o + 4])[0]
        assert np.array_equal(pool[o + M + 3 * (n + 1): o + M + 4 * (n + 1)], np.eye(n + 1)[3])
    forced = dict(tabs, pool=pool)
    E = emu_path_rows.PathRowsEmuEngine(P)
    E.set_path_rows(forced)
    lay = E.path_rows_layout()
    lost = sum(1 for k, i, nk, _ in P.aero_i32 if nk > 1 and i in moved)
    assert lost > 0 and lay["n_rows"] == 37 - lost
    assert not any(l == 3 and P.aero_i32[j, 1] in moved for j, l in zip(lay["job"], lay["l"]))
    assert list(zip(lay["job"], lay["l"])) == _want_layout(O, P, forced)
    x = helpers.perturbed(x0)
    g, v = E.eval_path_rows(problem.xdict_to_vector(x))
    gw, vw = path_rows_oracle.path_rows(O, x, forced)
    assert _eq(g, gw) and _eq(v, vw)


def _one_point_grid(tabs, ps, l):
    """Test point l of every section of `tabs` alone (tau_t, P and Q rows l, I = 1)."""
    parts, off, o = [], [], 0
    for i in range(ps.num_sections()):
        tau_t, P, Q, _ = mesh_oracle.unpack(tabs, i, ps.nodes(i))
        k = min(l, tau_t.size - 1)
        off.append(o)
        for a in (tau_t[k:k + 1], P[k], Q[k], np.ones(1)):
            parts.append(a.ravel())
            o += a.size
    return {"m": np.ones(ps.num_sections(), dtype=np.int32), "off": np.array(off, dtype=np.int64),
            "pool": np.concatenate(parts)}


@pytest.mark.parametrize("variant", ["example", "all_aero"])
def test_rows_are_the_path_check_residuals(variant):
    """Row (j, l) is the path check's residual at test point l, and the minimum over job j's rows and its last node
    row (the dropped point +1) is path_check's res[j], bit for bit."""
    p, u, c, x0, O, P = _setup(variant)
    E = emu_path_rows.PathRowsEmuEngine(P)
    tabs = mesh.grid_tables(O.ps)
    E.set_path_rows(tabs)
    E.set_mesh_grid(tabs)
    lay = E.path_rows_layout()
    for x in _points(x0, P, variant, 1):
        xv = problem.xdict_to_vector(x)
        g, _ = E.eval_path_rows(xv, jacobian=False)
        gn = E.eval_residuals(xv)
        res, at = E.path_check(xv)
        for j, (kind, i, nk, row0) in enumerate(P.aero_i32):
            if nk == 1:
                continue
            mine = lay["job"] == j
            both = np.append(g[mine], gn[row0 + nk - 1])
            assert _bits(both.min()) == _bits(res[j]), j
        for l in range(int(tabs["m"].max()) - 1):
            E.set_mesh_grid(_one_point_grid(tabs, O.ps, l))
            res1, _ = E.path_check(xv)
            for k in np.flatnonzero(lay["l"] == l):
                assert _bits(g[k]) == _bits(res1[lay["job"][k]]), (l, k)
        E.set_mesh_grid(tabs)


def _dense(blocks, rows, cols):
    """The entries of COO blocks [(rows, cols, values)] at (rows, cols) as a dense array."""
    D = np.zeros((len(rows), len(cols)))
    ri = {r: a for a, r in enumerate(rows)}
    ci = {c: b for b, c in enumerate(cols)}
    for r, c, d in blocks:
        for rr, cc, dd in zip(r, c, d):
            if rr in ri and cc in ci:
                D[ri[rr], ci[cc]] = dd
    return D


def _cd4(fun, x, cols, h):
    """4th-order central differences of fun(x)[rows] along the flat columns `cols` of x."""
    out = []
    for c in cols:
        vals = []
        for s in (2, 1, -1, -2):
            y = x.copy()
            y[c] += s * h
            vals.append(fun(y))
        out.append((-vals[0] + 8 * vals[1] - 8 * vals[2] + vals[3]) / (12 * h))
    return np.array(out).T


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("variant", ["example", "all_aero"])
def test_derivative_against_fourth_order_differences(variant, mode):
    """Per job and variable, the path rows' Jacobian is within a factor 10 as close to 4th-order differences of the
    oracle's path rows (perturbing x, step 1e-6) as the job's node rows are to theirs; closeness = the largest entry
    error over the largest true entry.  At the perturbed x0 the measured ratio is 0.3 to 5.8: the worst entries sit on
    the kinks of the piecewise-linear wind and CA tables, which neither quotient resolves, and the t blocks' true
    derivatives are at the quotients' noise level in both row sets."""
    p, u, c, x0, O, P = _setup(variant)
    E = emu_path_rows.PathRowsEmuEngine(P)
    tabs = mesh.grid_tables(O.ps)
    E.set_path_rows(tabs)
    E.set_fd(mode)
    lay = E.path_rows_layout()
    x = helpers.perturbed(x0)
    xv = problem.xdict_to_vector(x)
    _, pv = E.eval_path_rows(xv)
    st = P.path_rows_structure(lay)
    sj = P.split_jacobian(E.eval_jacobian(xv))
    off = P.off

    def path_g(y):
        return path_rows_oracle.path_rows(O, problem.vector_to_xdict(y, P.M, P.N, P.S), tabs, jacobian=False)[0]

    for j, (kind, i, nk, row0) in enumerate(P.aero_i32):
        if nk == 1:
            continue
        xa, n = P.ps.get_index(i)[2], P.ps.nodes(i)
        rows_p = list(np.flatnonzero(lay["job"] == j))
        grow0, _ = P.group_rows[AERO_KEYS[kind]]
        rows_n = list(range(row0 - grow0, row0 - grow0 + nk))
        for var, w in (("position", 3), ("velocity", 3), ("quaternion", 4), ("t", 1)):
            if var == "quaternion" and kind == 1:
                continue
            lc = [i, i + 1] if var == "t" else list(range(w * xa, w * (xa + n + 1)))
            gc = [off[var] + k for k in lc]
            b = st[var]
            Jp = _dense([(b.rows, b.cols, pv[b.offset:b.offset + b.nnz])], rows_p, lc)
            Tp = _cd4(lambda y: path_g(y)[rows_p], xv, gc, h=1e-6)
            bn = sj[AERO_KEYS[kind]][var]["coo"]
            Jn = _dense([bn], rows_n, lc)
            Tn = _cd4(lambda y: E.eval_residuals(y)[row0:row0 + nk], xv, gc, h=1e-6)
            ep = np.max(np.abs(Jp - Tp)) / np.max(np.abs(Tp))
            en = np.max(np.abs(Jn - Tn)) / np.max(np.abs(Tn))
            assert ep <= 10.0 * en, (j, var, ep, en)


def _problem(path_grid=None, **kw):
    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    prob = callbacks.GelatoProblem(p, u, c, user_eq=callbacks.PerigeeAtEvent(helpers.USER_EVENT), coord=Lg.coordinate_c,
                                   engine_factory=emu_path_rows.PathRowsEmuEngine, path_grid=path_grid, **kw)
    return prob, p, u, c, x0


def _sens_equal(sa, sb, keys):
    for k in keys:
        if sa[k] is None or sb[k] is None:
            assert sa[k] is None and sb[k] is None, k
            continue
        assert list(sa[k]) == list(sb[k]), k
        for var in sa[k]:
            a, b = sa[k][var], sb[k][var]
            if isinstance(a, dict):
                for q in range(3):
                    assert _eq(a["coo"][q], b["coo"][q]) if q == 2 else np.array_equal(a["coo"][q], b["coo"][q]), (k, var)
                assert a["shape"] == b["shape"]
            else:
                assert _eq(a, b), (k, var)


@pytest.mark.parametrize("kw", [{}, {"fuse_pair": True}, {"reuse_output": False}, {"derivative": "central"}])
def test_gelato_problem_with_and_without_path_grid(kw):
    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    tabs = mesh.grid_tables(p["ps_params"])
    base, _, _, _, _ = _problem(**kw)
    prob, _, _, _, _ = _problem(tabs, **kw)
    P = prob.plan
    O = helpers.oracle_nlp(p, u, c, "gmath", "seqfma")
    mode = kw.get("derivative", "forward")
    for x in (helpers.perturbed(x0), _solution(P)):
        f0, _ = base.objfunc(x)
        f1, _ = prob.objfunc(x)
        assert list(f1) == list(f0) + ["ineqcon_path"]
        for k in f0:
            assert (f0[k] is None and f1[k] is None) or _eq(f0[k], f1[k]), k
        s0, _ = base.sens(x, f0)
        s1, _ = prob.sens(x, f1)
        assert list(s1) == list(s0) + ["ineqcon_path"]
        _sens_equal(s0, s1, list(s0))
        gw, vw = path_rows_oracle.path_rows(O, x, tabs, mode)
        assert _eq(f1["ineqcon_path"], gw)
        blk = s1["ineqcon_path"]
        assert list(blk) == ["position", "velocity", "quaternion", "t"]
        assert _eq(np.concatenate([blk[v]["coo"][2] for v in blk]), vw)
        if prob.reuse_output:  # the data arrays are views of one kept buffer
            bases = {b["coo"][2].base is not None and id(b["coo"][2].base) for b in blk.values()}
            assert len(bases) == 1 and False not in bases
        # jacobian_csr: the registered groups, then the path rows, equal to the stacked COO
        J = prob.jacobian_csr(x)
        Jb = base.jacobian_csr(x)
        nr = len(gw)
        assert J.shape == (Jb.shape[0] + nr, Jb.shape[1])
        assert (J[:Jb.shape[0]] != Jb).nnz == 0
        import scipy.sparse as sp

        col0 = dict(zip(callbacks.VAR_ORDER, np.cumsum([0] + [P.sizes[k] for k in callbacks.VAR_ORDER])))
        coo = sp.coo_matrix((np.concatenate([blk[v]["coo"][2] for v in blk]),
                             (np.concatenate([blk[v]["coo"][0] for v in blk]),
                              np.concatenate([np.asarray(blk[v]["coo"][1], dtype=np.int64) + col0[v] for v in blk]))),
                            shape=(nr, Jb.shape[1]))
        assert (J[Jb.shape[0]:] != coo.tocsr()).nnz == 0
    idx = prob.path_rows_index()
    assert len(idx) == 16 and all(k == ("ineqcon_qalpha", "ZEROLIFT_START") for k, _, _ in [(a[:2], 0, 0) for a in idx])
    assert [a[2] for a in idx] == list(range(16)) and base.path_rows_index() == []
    # registration: nlpshim.register takes the group like any other inequality
    opt = nlpshim.register(prob.objfunc, prob.sens, x0, c)
    names = [g[0] for g in opt.cons]
    assert names[-1] == "ineqcon_path" and opt.cons[-1][1] == 16 and opt.cons[-1][2] == 0.0 and opt.cons[-1][3] is None
    assert opt.cons[-1][4] == ["position", "velocity", "quaternion", "t"]
    assert names[:-1] == [g[0] for g in nlpshim.register(base.objfunc, base.sens, x0, c).cons]
    base.close()
    prob.close()


def test_fused_pair_keeps_the_path_rows_jacobian():
    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    prob, _, _, _, _ = _problem(mesh.grid_tables(p["ps_params"]), fuse_pair=True)
    x = helpers.perturbed(x0)
    f, _ = prob.objfunc(x)
    calls = prob.engine.calls
    s, _ = prob.sens(x, f)
    assert prob.engine.calls == calls  # neither Jacobian is evaluated again
    O = helpers.oracle_nlp(p, u, c, "gmath", "seqfma")
    assert _eq(np.concatenate([b["coo"][2] for b in s["ineqcon_path"].values()]),
               path_rows_oracle.path_rows(O, x, mesh.grid_tables(p["ps_params"]))[1])
    prob.close()


def test_refusals():
    p, u, c, x0, O, P = _setup("example")
    E = emu_path_rows.PathRowsEmuEngine(P)
    xv = problem.xdict_to_vector(x0)
    with pytest.raises(engine.GelatoError, match="no path rows set"):
        E.eval_path_rows(xv)
    with pytest.raises(engine.GelatoError, match="no path rows set"):
        E.path_rows_layout()
    tabs = mesh.grid_tables(O.ps)
    E.set_path_rows(tabs)
    ref = E.eval_path_rows(xv)
    bad = dict(tabs, pool=tabs["pool"].copy())
    bad["pool"][5] = np.nan
    with pytest.raises(engine.GelatoError, match="not finite"):
        E.set_path_rows(bad)
    with pytest.raises(engine.GelatoError, match="at least one test point"):
        E.set_path_rows(dict(tabs, m=np.zeros_like(tabs["m"])))
    got = E.eval_path_rows(xv)  # the refused grids left the rows as they were
    assert _eq(got[0], ref[0]) and _eq(got[1], ref[1])
    # a bare plan: zero rows, nothing written
    p, u, c, x0, O, P = _setup("bare")
    E = emu_path_rows.PathRowsEmuEngine(P)
    E.set_path_rows(mesh.grid_tables(O.ps))
    lay = E.path_rows_layout()
    assert (lay["n_rows"], lay["n_vals"]) == (0, 0)
    g, v = E.eval_path_rows(problem.xdict_to_vector(x0))
    assert g.shape == (0,) and v.shape == (0,)
    assert path_rows_oracle.path_rows(O, x0, mesh.grid_tables(O.ps))[0].shape == (0,)


@pytest.mark.parametrize("case", edge.CASES)
@pytest.mark.parametrize("variant", ["example", "all_aero"])
def test_edge_states(variant, case):
    """The edge-state catalogue of test_edge_states: equal bits, or NaN on both sides."""
    p, u, c, x0, O, P = edge._setup(variant)
    E = emu_path_rows.PathRowsEmuEngine(P)
    tabs = mesh.grid_tables(P.ps)
    E.set_path_rows(tabs)
    x = edge.CATALOGUE[case][0](x0, P)
    xv = problem.xdict_to_vector(x)
    for mode in (MODES if case in edge.CENTRAL_CASES else MODES[:1]):
        E.set_fd(mode)
        g, v = E.eval_path_rows(xv)
        with np.errstate(all="ignore"):
            gw, vw = path_rows_oracle.path_rows(O, x, tabs, mode)
        for a, b in ((g, gw), (v, vw)):
            ok, why = edge._same(a, b)
            assert ok, (mode, why)


# ------------------------------------------------------------------------------------------------ GPU tier
def _engine(P, scenario_plans=None):
    return engine.Engine(P, device=0, scenario_plans=scenario_plans)


@pytest.mark.gpu
@pytest.mark.parametrize("variant,factor", VARIANTS)
def test_gpu_equals_oracle_bit_for_bit(variant, factor):
    p, u, c, x0, O, P = _setup(variant, factor)
    E = _engine(P)
    for tabs in _grids(O.ps):
        E.set_path_rows(tabs)
        lay = E.path_rows_layout()
        assert list(zip(lay["job"], lay["l"])) == _want_layout(O, P, tabs)
        for mode in MODES:
            E.set_fd(mode)
            for x in _points(x0, P, variant, factor):
                xv = problem.xdict_to_vector(x)
                g, v = E.eval_path_rows(xv)
                gw, vw = path_rows_oracle.path_rows(O, x, tabs, mode)
                assert _eq(g, gw) and _eq(v, vw), mode
                g1, v1 = E.eval_path_rows(xv, jacobian=False)
                assert v1 is None and _eq(g1, g)  # residual only: the same g
    E.close()


@pytest.mark.gpu
def test_gpu_dispersed_batch_with_per_scenario_blocks():
    Lg = leaves.get("gmath")
    scen = scenarios.disperse(helpers.example_inputs(), 64, seed=11)
    plans, xs, oracles = [], [], []
    for k, inp in enumerate(scen):
        p, u, c, x0 = problem.problem_from_inputs(inp, coord=Lg.coordinate_c)
        plans.append(helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c))
        xs.append(helpers.perturbed(x0, seed=k))
        oracles.append(helpers.oracle_nlp(p, u, c, "gmath", "seqfma"))
    E = _engine(plans[0], scenario_plans=plans)
    tabs = mesh.grid_tables(plans[0].ps)
    E.set_path_rows(tabs)
    X = np.stack([problem.xdict_to_vector(x) for x in xs])
    for mode in MODES:
        E.set_fd(mode)
        g, v = E.eval_path_rows(X, n_scen=64)
        assert g.shape == (64, 16) and v.shape == (64, 2752)
        for k in range(64):
            gw, vw = path_rows_oracle.path_rows(oracles[k], xs[k], tabs, mode)
            assert _eq(g[k], gw) and _eq(v[k], vw), (mode, k)
        g1, _ = E.eval_path_rows(X, n_scen=64, jacobian=False)
        assert _eq(g1, g)
    assert not _eq(g[0], g[1])
    with pytest.raises(engine.GelatoError, match="configured"):
        E.eval_path_rows(np.concatenate([X, X[:1]]), n_scen=65)
    E.close()


@pytest.mark.gpu
def test_gpu_bench_workload_sample():
    import bench

    Lg = leaves.get("gmath")
    plans, X, probs = bench.load_workload("example", 15, 128, 0, 128, coord=Lg.coordinate_c)
    E = _engine(plans[0], scenario_plans=plans)
    tabs = mesh.grid_tables(plans[0].ps)
    E.set_path_rows(tabs)
    lay = E.path_rows_layout()
    assert (lay["n_rows"], lay["n_vals"]) == (240, 50880)
    g, v = E.eval_path_rows(X, n_scen=128)
    assert g.shape == (128, 240) and not np.isnan(g).any() and not np.isnan(v).any()
    for k in (0, 37, 127):
        p, u, c, x = probs[k]
        gw, vw = path_rows_oracle.path_rows(helpers.oracle_nlp(p, u, c, "gmath", "seqfma"), x, tabs)
        assert _eq(g[k], gw) and _eq(v[k], vw), k
    E.close()


@pytest.mark.gpu
def test_gpu_host_pinned_dev_and_residual_only_agree():
    import torch

    p, u, c, x0, O, P = _setup("all_aero", 2)
    E = _engine(P, scenario_plans=[P] * 3)
    E.set_path_rows(mesh.grid_tables(O.ps))
    lay = E.path_rows_layout()
    nr, nv = lay["n_rows"], lay["n_vals"]
    X = np.stack([problem.xdict_to_vector(helpers.perturbed(x0, seed=k)) for k in range(3)])
    E.set_fd("central")
    ref = E.eval_path_rows(X, n_scen=3)
    px, pg, pvv = engine.PinnedArray(X.size), engine.PinnedArray(3 * nr), engine.PinnedArray(3 * nv)
    px.array[:] = X.ravel()
    E.eval_path_rows(px.array, n_scen=3, out=(pg.array, pvv.array))
    assert _eq(pg.array.reshape(3, nr), ref[0]) and _eq(pvv.array.reshape(3, nv), ref[1])
    xd = torch.from_numpy(X).cuda()
    gd = torch.full((3, nr), float("nan"), dtype=torch.float64, device="cuda")
    vd = torch.full((3, nv), float("nan"), dtype=torch.float64, device="cuda")
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        E.eval_path_rows_dev(xd.data_ptr(), gd.data_ptr(), vd.data_ptr(), 3, st.cuda_stream)
    st.synchronize()
    assert _eq(gd.cpu().numpy(), ref[0]) and _eq(vd.cpu().numpy(), ref[1])
    gd.fill_(float("nan"))
    E.eval_path_rows_dev(xd.data_ptr(), gd.data_ptr(), None, 3, None)  # residual only, the plan's stream
    torch.cuda.synchronize()
    assert _eq(gd.cpu().numpy(), ref[0])
    vd.fill_(float("nan"))
    E.eval_path_rows_dev(xd.data_ptr(), None, vd.data_ptr(), 3, None)  # Jacobian only
    torch.cuda.synchronize()
    assert _eq(vd.cpu().numpy(), ref[1])
    g1, v1 = E.eval_path_rows(X[1], jacobian=False)
    assert _eq(g1, ref[0][1]) and v1 is None
    for a in (px, pg, pvv):
        a.free()
    E.close()


@pytest.mark.gpu
def test_gpu_refusals_and_a_bare_plan():
    p, u, c, x0, O, P = _setup("example")
    E = _engine(P)
    xv = problem.xdict_to_vector(x0)
    with pytest.raises(engine.GelatoError, match="no path rows set"):
        E.eval_path_rows(xv)
    L = E.L
    n, v = ctypes.c_int32(0), ctypes.c_int64(0)
    assert L.gelato_plan_path_rows(E.h, ctypes.byref(n), ctypes.byref(v), None, None, None) == -1
    tabs = mesh.grid_tables(O.ps)
    E.set_path_rows(tabs)
    ref = E.eval_path_rows(xv)
    bad = dict(tabs, pool=tabs["pool"].copy())
    bad["pool"][5] = np.inf
    with pytest.raises(engine.GelatoError, match="not finite"):
        E.set_path_rows(bad)
    n, v = ctypes.c_int32(0), ctypes.c_int64(0)
    assert L.gelato_plan_path_rows(E.h, ctypes.byref(n), ctypes.byref(v), None, None, None) == 0
    assert (n.value, v.value) == (16, 2752)  # the refused grid changed nothing
    got = E.eval_path_rows(xv)
    assert _eq(got[0], ref[0]) and _eq(got[1], ref[1])
    xp = xv.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    assert L.gelato_eval_path_rows(E.h, xp, None, None, 0) == -1
    assert L.gelato_eval_path_rows(E.h, None, None, None, 1) == -1
    E.close()
    p, u, c, x0, O, P = _setup("bare")
    E = _engine(P)
    E.set_path_rows(mesh.grid_tables(O.ps))
    g, v = E.eval_path_rows(problem.xdict_to_vector(x0))
    assert g.shape == (0,) and v.shape == (0,)
    E.close()


@pytest.mark.gpu
def test_gpu_gelato_problem_with_path_grid_matches_the_emulator():
    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    tabs = mesh.grid_tables(p["ps_params"])
    gpu = callbacks.GelatoProblem(p, u, c, user_eq=callbacks.PerigeeAtEvent(helpers.USER_EVENT), coord=Lg.coordinate_c,
                                  device=0, path_grid=tabs, fuse_pair=True)
    emu, _, _, _, _ = _problem(tabs, fuse_pair=True)
    x = helpers.perturbed(x0)
    fg, _ = gpu.objfunc(x)
    fe, _ = emu.objfunc(x)
    assert list(fg) == list(fe) and all((fg[k] is None) or _eq(fg[k], fe[k]) for k in fg)
    sg, _ = gpu.sens(x, fg)
    se, _ = emu.sens(x, fe)
    _sens_equal(sg, se, [k for k in GROUPS if k != "eqcon_user"] + ["ineqcon_path"])
    gpu.close()
    emu.close()
