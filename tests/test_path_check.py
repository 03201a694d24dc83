"""Path check: the aero constraints between the collocation nodes (DESIGN.md section 11).

CPU tier: the kernels' code in the host emulator against the oracle bit for bit (variants, both grids, three decision
vectors), a plan without aero jobs, test points that are nodes against objfunc's own rows, the example solution's
violation between the nodes, refine_nodes with `path`, GelatoProblem.path_check and the refusal before a grid is set.
GPU tier: the C ABI against the oracle bit for bit (variants, a dispersed batch with per-scenario blocks, the benchmark
workload), host / device entry points and buffers, argument errors and the independence from the finite-difference
mode."""
import ctypes

import numpy as np
import pytest

import emu_path
import helpers
import mesh_oracle
import path_oracle
from gelato_b200 import callbacks, engine, mesh, problem, scenarios
from oracle import leaves

VARIANTS = [("example", 1), ("all_aero", 1), ("three_stage", 1), ("neg_area", 1), ("example", 15)]


def _bits(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64)).view(np.int64)


def _same(got, want):
    """(res, at) pairs equal bit for bit."""
    return (np.shape(got[0]) == np.shape(want[0]) and np.array_equal(_bits(got[0]), _bits(want[0]))
            and np.array_equal(np.asarray(got[1]), np.asarray(want[1])))


def _setup(variant, factor=1):
    Lg = leaves.get("gmath")
    p, u, c, x0 = problem.problem_from_inputs(helpers.variant_inputs(variant), coord=Lg.coordinate_c, factor=factor,
                                              max_nodes=20)
    O = helpers.oracle_nlp(p, u, c, "gmath", "seqfma")
    return p, u, c, x0, O, helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c)


def _solution(P):
    x = np.load(helpers.GOLDEN + "/example_solution.npz")["x"]
    return problem.vector_to_xdict(x, P.M, P.N, P.S)


def _points(x0, P, variant, factor):
    return [x0, helpers.perturbed(x0)] + ([_solution(P)] if (variant, factor) == ("example", 1) else [])


def _square_grid(ps):
    return mesh.grid_tables(ps, m=[ps.nodes(i) for i in range(ps.num_sections())])


def _node_grid(ps, l):
    """One test point per section: its LGR node min(l, n - 1) (tau_t = tau_l, P = the identity row)."""
    parts, off, o = [], [], 0
    for i in range(ps.num_sections()):
        tau = ps.tau(i)
        n = tau.size
        tt = tau[min(l, n - 1):][:1]
        P = mesh.lagrange_basis(np.hstack((-1.0, tau)), tt)
        assert np.array_equal(P, np.eye(n + 1)[min(l, n - 1) + 1:][:1])
        Q = mesh.lagrange_basis(tau, tt)
        off.append(o)
        for a in (tt, P, Q, np.ones((1, 1))):
            parts.append(a.ravel())
            o += a.size
    return {"m": np.ones(ps.num_sections(), dtype=np.int32), "off": np.array(off, dtype=np.int64),
            "pool": np.concatenate(parts)}


def _job(P, kind, name):
    """Index of the aero job of `kind` (0 alpha, 1 q, 2 Q-alpha) over the section of event `name`."""
    i = P.p["event_index"][name]
    return [j for j, a in enumerate(P.aero_i32) if a[0] == kind and a[1] == i][0]


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("variant,factor", VARIANTS)
def test_emulator_equals_oracle_bit_for_bit(variant, factor):
    p, u, c, x0, O, P = _setup(variant, factor)
    E = emu_path.PathEmuEngine(P)
    assert P.n_aero > 0
    for tabs in (mesh.grid_tables(O.ps), _square_grid(O.ps)):
        E.set_mesh_grid(tabs)
        for x in _points(x0, P, variant, factor):
            got = E.path_check(problem.xdict_to_vector(x))
            assert got[0].shape == (P.n_aero,) and got[1].dtype == np.int32
            assert _same(got, path_oracle.path_check(O, x, tabs))


def test_all_aero_has_every_kind_and_both_ranges():
    p, u, c, x0, O, P = _setup("all_aero")
    assert {int(k) for k in P.aero_i32[:, 0]} == {0, 1, 2}
    assert {int(k) for k, _, nk, _ in P.aero_i32 if nk == 1} == {0, 1, 2}  # "initial" jobs
    assert {int(k) for k, _, nk, _ in P.aero_i32 if nk > 1} == {0, 1, 2}  # "all" jobs
    E = emu_path.PathEmuEngine(P)
    E.set_mesh_grid(mesh.grid_tables(O.ps))
    res, at = E.path_check(problem.xdict_to_vector(helpers.perturbed(x0)))
    initial = P.aero_i32[:, 2] == 1
    assert np.all(res[initial] == np.inf) and np.all(at[initial] == -1)
    assert np.isfinite(res[~initial]).all() and np.all(at[~initial] >= 0)


def test_bare_plan_has_no_aero_jobs_and_an_empty_result():
    p, u, c, x0, O, P = _setup("bare")
    assert P.n_aero == 0
    E = emu_path.PathEmuEngine(P)
    E.set_mesh_grid(mesh.grid_tables(O.ps))
    res, at = E.path_check(problem.xdict_to_vector(x0))
    assert res.shape == (0,) and at.shape == (0,)
    res, at = E.path_check(np.stack([problem.xdict_to_vector(x0)] * 2), n_scen=2)
    assert res.shape == (2, 0) and at.shape == (2, 0)
    assert _same(path_oracle.path_check(O, x0, mesh.grid_tables(O.ps)), (np.zeros(0), np.zeros(0, dtype=np.int32)))


@pytest.mark.parametrize("variant", ["example", "all_aero", "three_stage"])
def test_test_points_at_nodes_are_objfunc_rows(variant):
    """A test point that is an LGR node gives objfunc's row there bit for bit: one node per section at a time, the square
    grid (the minimum of the job's node rows after the first) and the default grid's last point (the job's last row)."""
    p, u, c, x0, O, P = _setup(variant)
    E = emu_path.PathEmuEngine(P)
    x = helpers.perturbed(x0)
    xv = problem.xdict_to_vector(x)
    g = E.eval_residuals(xv)
    full = P.aero_i32[:, 2] > 1
    assert full.any()
    for l in range(max(O.ps.nodes(i) for i in range(O.S))):
        E.set_mesh_grid(_node_grid(O.ps, l))
        res, at = E.path_check(xv)
        for j, (kind, i, nk, row0) in enumerate(P.aero_i32):
            if nk > 1:
                assert _bits(res[j]) == _bits(g[row0 + min(l, nk - 2) + 1]) and at[j] == 0, (l, j)
    E.set_mesh_grid(_square_grid(O.ps))
    res, at = E.path_check(xv)
    for j, (kind, i, nk, row0) in enumerate(P.aero_i32):
        if nk > 1:
            rows = g[row0 + 1:row0 + nk]
            assert _bits(res[j]) == _bits(rows.min()) and at[j] == int(np.argmin(rows)), j
    E.set_mesh_grid(mesh.grid_tables(O.ps, m=1))  # the one flipped LGR point of one node: +1
    res, at = E.path_check(xv)
    for j, (kind, i, nk, row0) in enumerate(P.aero_i32):
        if nk > 1:
            assert _bits(res[j]) == _bits(g[row0 + nk - 1]) and at[j] == 0, j


def test_example_solution_violates_q_alpha_between_the_nodes():
    """The converged example holds Q-alpha at ZEROLIFT_START's nodes and exceeds it by 6 % in between."""
    p, u, c, x0, O, P = _setup("example")
    E = emu_path.PathEmuEngine(P)
    tabs = mesh.grid_tables(O.ps)
    E.set_mesh_grid(tabs)
    x = _solution(P)
    xv = problem.xdict_to_vector(x)
    res, at = E.path_check(xv)
    j = _job(P, 2, "ZEROLIFT_START")
    i = P.aero_i32[j, 1]
    assert -6.12e-2 < res[j] < -6.10e-2
    tau_t = mesh_oracle.unpack(tabs, i, O.ps.nodes(i))[0]
    assert abs(tau_t[at[j]] - (-0.137)) < 1e-3
    kind, _, nk, row0 = P.aero_i32[j]
    assert np.all(E.eval_residuals(xv)[row0:row0 + nk] >= 0.0)  # what the solver saw
    m = _job(P, 0, "MECO")  # "initial": a point constraint
    assert P.aero_i32[m, 2] == 1 and res[m] == np.inf and at[m] == -1


def test_emulator_refuses_a_call_before_a_grid_is_set():
    p, u, c, x0, O, P = _setup("example")
    E = emu_path.PathEmuEngine(P)
    with pytest.raises(engine.GelatoError, match="no mesh grid set"):
        E.path_check(problem.xdict_to_vector(x0))


def test_refine_nodes_with_path_rule_cap_and_unchanged_without_it():
    ev = helpers.example_inputs()["events"]
    S = len(ev) - 1
    err = np.zeros((S, 11))
    err[0, 3] = 1e-3  # LIFTOFF, n = 5: 5 + ceil(log(1e4) / log(5)) = 11
    err[4, 1] = 1e-7  # MECO: equal to tol, untouched
    base, rep0 = mesh.refine_nodes(ev, err, tol=1e-7, n_max=12)
    same, rep1 = mesh.refine_nodes(ev, err, tol=1e-7, n_max=12, path=None)
    assert same == base and rep1 == rep0 and all(r.path is None for r in rep0)
    assert [r.n_new for r in rep0][:3] == [11, 5, 16]
    path = np.full(S, np.inf)
    path[0] = -1e-2   # LIFTOFF: 5 + ceil(log(10) / log(5)) = 7 < 11 from the estimate: 11
    path[1] = -5e-2   # KICKTURN, n = 5: 5 + ceil(log(50) / log(5)) = 8
    path[2] = -6e-2   # ZEROLIFT_START, n = 16 > n_max: not split, reported
    path[3] = -1e-3   # ZEROLIFT_END: equal to -path_tol, untouched
    path[5] = 0.5     # satisfied
    path[6] = -1e4    # SEIG, n = 5: 5 + ceil(log(1e7) / log(5)) = 16, capped at 12
    new, rep = mesh.refine_nodes(ev, err, tol=1e-7, n_max=12, path=path, path_tol=1e-3)
    got = {r.name: (r.n_old, r.n_new, r.capped, r.path) for r in rep}
    assert got["LIFTOFF"] == (5, 11, False, -1e-2)
    assert got["KICKTURN"] == (5, 8, False, -5e-2)
    assert got["ZEROLIFT_START"] == (16, 16, True, -6e-2)
    assert got["ZEROLIFT_END"] == (8, 8, False, -1e-3)
    assert got["SEIG"] == (5, 12, True, -1e4)
    assert got["MECO"][3] is None and got["FAIRING"][1:] == (6, False, None)
    assert [e["num_nodes"] for e in new[:S]] == [r.n_new for r in rep]
    # the dictionary of GelatoProblem.path_check: the worst entry of a section counts
    d = {("ineqcon_qalpha", "KICKTURN"): (-5e-2, 10.0), ("ineqcon_alpha", "KICKTURN"): (0.1, 12.0),
         ("ineqcon_q", "SEIG"): (-2e-3, 400.0)}
    new2, rep2 = mesh.refine_nodes(ev, np.zeros((S, 11)), tol=1e-7, n_max=12, path=d)
    got = {r.name: (r.n_new, r.path) for r in rep2}
    assert got["KICKTURN"] == (8, -5e-2) and got["SEIG"] == (6, -2e-3) and got["LIFTOFF"] == (5, None)
    for bad in (np.full(S, np.nan), np.full(S, -np.inf)):
        with pytest.raises(ValueError):
            mesh.refine_nodes(ev, err, tol=1e-7, n_max=12, path=bad)


def test_gelato_problem_path_check_on_the_emulator():
    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    prob = callbacks.GelatoProblem(p, u, c, user_eq=callbacks.PerigeeAtEvent(helpers.USER_EVENT), coord=Lg.coordinate_c,
                                   engine_factory=emu_path.PathEmuEngine)
    P = prob.plan
    x = _solution(P)
    got = prob.path_check(x)
    tabs = mesh.grid_tables(p["ps_params"])
    res, at = path_oracle.path_check(helpers.oracle_nlp(p, u, c, "gmath", "seqfma"), x, tabs)
    full = [j for j in range(P.n_aero) if P.aero_i32[j, 2] > 1]
    assert list(got) == [(("ineqcon_alpha", "ineqcon_q", "ineqcon_qalpha")[P.aero_i32[j, 0]],
                          p["params"][P.aero_i32[j, 1]]["name"]) for j in full]
    r, t_s = got[("ineqcon_qalpha", "ZEROLIFT_START")]
    j = _job(P, 2, "ZEROLIFT_START")
    i = P.aero_i32[j, 1]
    assert _bits(r) == _bits(res[j])
    tau = mesh_oracle.unpack(tabs, i, p["ps_params"].nodes(i))[0][at[j]]
    to, tf = x["t"][i], x["t"][i + 1]
    assert t_s == (tau * (tf - to) / 2 + (tf + to) / 2) * u["t"] and to * u["t"] < t_s < tf * u["t"]
    assert prob.mesh_error(x).keys() and prob.path_check(x) == got  # the grid is shared and set once
    new, rep = mesh.refine_nodes(helpers.example_inputs()["events"], prob.mesh_error(x), 1e-6, 30, path=got)
    assert {r.name: r.n_new for r in rep}["ZEROLIFT_START"] > 16
    prob.close()


# ------------------------------------------------------------------------------------------------ GPU tier
def _engine(P, scenario_plans=None):
    return engine.Engine(P, device=0, scenario_plans=scenario_plans)


@pytest.mark.gpu
@pytest.mark.parametrize("variant,factor", VARIANTS)
def test_gpu_equals_oracle_bit_for_bit(variant, factor):
    p, u, c, x0, O, P = _setup(variant, factor)
    E = _engine(P)
    for tabs in (mesh.grid_tables(O.ps), _square_grid(O.ps)):
        E.set_mesh_grid(tabs)
        for x in _points(x0, P, variant, factor):
            assert _same(E.path_check(problem.xdict_to_vector(x)), path_oracle.path_check(O, x, tabs))
    E.close()


@pytest.mark.gpu
def test_gpu_bare_plan_returns_empty_results():
    p, u, c, x0, O, P = _setup("bare")
    E = _engine(P)
    E.set_mesh_grid(mesh.grid_tables(O.ps))
    res, at = E.path_check(problem.xdict_to_vector(x0))
    assert res.shape == (0,) and at.shape == (0,)
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
    E.set_mesh_grid(tabs)
    res, at = E.path_check(np.stack([problem.xdict_to_vector(x) for x in xs]), n_scen=64)
    assert res.shape == (64, plans[0].n_aero)
    for k in range(64):
        assert _same((res[k], at[k]), path_oracle.path_check(oracles[k], xs[k], tabs)), k
    full = plans[0].aero_i32[:, 2] > 1
    assert not np.array_equal(_bits(res[0][full]), _bits(res[1][full]))  # the per-scenario blocks are read
    E.close()


@pytest.mark.gpu
def test_gpu_bench_workload_sample():
    import bench

    Lg = leaves.get("gmath")
    plans, X, probs = bench.load_workload("example", 15, 128, 0, 128, coord=Lg.coordinate_c)
    E = _engine(plans[0], scenario_plans=plans)
    tabs = mesh.grid_tables(plans[0].ps)
    E.set_mesh_grid(tabs)
    res, at = E.path_check(X, n_scen=128)
    assert res.shape == (128, plans[0].n_aero) and not np.isnan(res).any()
    for k in (0, 37, 127):
        p, u, c, x = probs[k]
        assert _same((res[k], at[k]), path_oracle.path_check(helpers.oracle_nlp(p, u, c, "gmath", "seqfma"), x, tabs)), k
    E.close()


@pytest.mark.gpu
def test_gpu_host_dev_pinned_pageable_agree():
    import torch

    p, u, c, x0, O, P = _setup("all_aero", 2)
    E = _engine(P, scenario_plans=[P] * 3)
    E.set_mesh_grid(mesh.grid_tables(O.ps))
    X = np.stack([problem.xdict_to_vector(helpers.perturbed(x0, seed=k)) for k in range(3)])
    ref = E.path_check(X, n_scen=3)
    n = ref[0].size
    px, pr, pa = engine.PinnedArray(X.size), engine.PinnedArray(n), engine.PinnedArray(n)
    px.array[:] = X.ravel()
    at_pinned = pa.array.view(np.int32)[:n]
    E.path_check(px.array, n_scen=3, out=(pr.array, at_pinned))
    assert _same((pr.array.reshape(ref[0].shape), at_pinned.reshape(ref[1].shape)), ref)
    xd = torch.from_numpy(X).cuda()
    rd = torch.full(ref[0].shape, float("nan"), dtype=torch.float64, device="cuda")
    ad = torch.full(ref[1].shape, -2, dtype=torch.int32, device="cuda")
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        E.path_check_dev(xd.data_ptr(), rd.data_ptr(), ad.data_ptr(), 3, st.cuda_stream)
    st.synchronize()
    assert _same((rd.cpu().numpy(), ad.cpu().numpy()), ref)
    assert _same(E.path_check(X[1]), (ref[0][1], ref[1][1]))  # a smaller batch after a larger one
    for a in (px, pr, pa):
        a.free()
    E.close()


@pytest.mark.gpu
def test_gpu_argument_errors_leave_the_plan_usable_and_fd_mode_is_irrelevant():
    p, u, c, x0, O, P = _setup("example", 1)
    E = _engine(P)
    x = problem.xdict_to_vector(helpers.perturbed(x0))
    with pytest.raises(engine.GelatoError, match="no mesh grid"):
        E.path_check(x)
    E.set_mesh_grid(mesh.grid_tables(O.ps))
    ref = E.path_check(x)
    L = E.L
    res, at = np.empty(P.n_aero), np.empty(P.n_aero, dtype=np.int32)
    xp = x.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    rp = res.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    ap = at.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
    assert L.gelato_eval_path_check(E.h, xp, rp, ap, 0) == -1
    assert L.gelato_eval_path_check(E.h, None, rp, ap, 1) == -1
    assert L.gelato_eval_path_check(E.h, xp, rp, None, 1) == -1
    assert _same(E.path_check(x), ref)
    E.set_fd("central")
    E.eval_jacobian(x)
    assert _same(E.path_check(x), ref)
    E.close()
    # per-scenario blocks: an n_scen beyond the configured scenarios is refused
    E2 = _engine(P, scenario_plans=[P, P])
    E2.set_mesh_grid(mesh.grid_tables(O.ps))
    with pytest.raises(engine.GelatoError, match="configured"):
        E2.path_check(np.stack([x] * 3), n_scen=3)
    got = E2.path_check(np.stack([x] * 2), n_scen=2)
    assert _same((got[0][1], got[1][1]), ref)
    E2.close()
