"""Mesh error estimate, p-refinement and solution transfer (DESIGN.md section 11).

CPU tier: the tables of gelato_b200.mesh, the oracle's estimate on each section's own grid against -A^-1 g (g =
objfunc's collocation defect), the kernels' code in the host emulator against the oracle bit for bit, the convergence
of the estimate on the example's vacuum coast sections for a state integrated to high accuracy, refine_nodes,
transfer and GelatoProblem.mesh_error on the emulator.  GPU tier: the C ABI against the oracle bit for bit (variants,
a dispersed batch with per-scenario blocks, the benchmark workload), the square grid against the GPU's own defects,
host / device entry points and buffers, argument errors and the independence from the finite-difference mode."""
import ctypes

import numpy as np
import pytest

import helpers
import mesh_oracle
from emu_mesh import MeshEmuEngine
from gelato_b200 import callbacks, engine, mesh, problem, scenarios
from gelato_b200.psparams import PSparams, lgr_diff_matrix, lgr_nodes
from oracle import leaves

EPS = np.finfo(np.float64).eps
VARIANTS = [("example", 1), ("three_stage", 1), ("neg_area", 1), ("example", 15)]


def _bits(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64)).view(np.int64)


def _same_bits(a, b):
    return np.asarray(a).shape == np.asarray(b).shape and np.array_equal(_bits(a), _bits(b))


def _setup(variant, factor=1):
    Lg = leaves.get("gmath")
    p, u, c, x0 = problem.problem_from_inputs(helpers.variant_inputs(variant), coord=Lg.coordinate_c, factor=factor,
                                              max_nodes=20)
    O = helpers.oracle_nlp(p, u, c, "gmath", "seqfma")
    return p, u, c, x0, O, helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c)


def _solution(P):
    x = np.load(helpers.GOLDEN + "/example_solution.npz")["x"]
    return problem.vector_to_xdict(x, P.M, P.N, P.S)


def _square_grid(ps):
    return mesh.grid_tables(ps, m=[ps.nodes(i) for i in range(ps.num_sections())])


def _defects(O, g):
    """Per section, g_defect[n][11] (mass | position | velocity | quaternion) from a residual dictionary."""
    out = []
    for i in range(O.S):
        ua, ub, xa, xb, n = O.ps.get_index(i)
        out.append(np.column_stack((g["eqcon_dyn_mass"][ua:ub], g["eqcon_dyn_pos"].reshape(-1, 3)[ua:ub],
                                    g["eqcon_dyn_vel"].reshape(-1, 3)[ua:ub], g["eqcon_dyn_quat"].reshape(-1, 4)[ua:ub])))
    return out


def _check_square_grid(O, x, err, g):
    """err (the estimate on each section's own grid) against -A^-1 g for the D.X rows and -g for the difference rows;
    the bound of the D.X rows is the rounding of the two computations carried through A^-1."""
    for i, gd in enumerate(_defects(O, g)):
        n = O.ps.nodes(i)
        prm = O.p["params"][i]
        X, _ = mesh_oracle.section_states(O, x, i)
        A = lgr_diff_matrix(n)[:, 1:]
        Ainv = np.linalg.inv(A)
        scale = 1.0 + np.max(np.abs(X[1:]), axis=0)
        diff_rows = [0] * (not prm["engineOn"]) + [7, 8, 9, 10] * O._holds(i)
        for c in range(11):
            if c in diff_rows:
                assert err[i, c] == np.max(np.abs(gd[:, c])) / scale[c], (i, c)
                continue
            want = np.max(np.abs(Ainv @ gd[:, c])) / scale[c]
            D = lgr_diff_matrix(n)
            rh = D @ X[:, c] - gd[:, c]
            ulp = (n + 3) * EPS * (np.abs(D) @ np.abs(X[:, c]) + np.abs(rh) + np.abs(X[1:, c]))
            bound = 8.0 * (np.abs(Ainv).sum(axis=1).max() * ulp.max() + (n + 3) * EPS * np.max(np.abs(X[:, c]))) / scale[c]
            assert abs(err[i, c] - want) <= bound, (i, c, err[i, c], want, bound)


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("n", [2, 5, 12, 20])
def test_tables_are_exact_on_polynomials_and_on_coincident_points(n):
    tau = lgr_nodes(n)
    s = np.hstack((-1.0, tau))
    rng = np.random.default_rng(n)
    for m in (n - 1, n, n + 1, 2 * n):
        tt, P, Q, I = mesh.section_tables(tau, m)
        cx, cu, ci = rng.normal(size=n + 1), rng.normal(size=n), rng.normal(size=m)
        assert np.allclose(P @ np.polyval(cx, s), np.polyval(cx, tt), rtol=0, atol=1e-12 * np.abs(cx).sum())
        assert np.allclose(Q @ np.polyval(cu, tau), np.polyval(cu, tt), rtol=0, atol=1e-12 * np.abs(cu).sum())
        F = np.polyint(ci)  # the integral from -1 of a degree m - 1 polynomial
        assert np.allclose(I @ np.polyval(ci, tt), np.polyval(F, tt) - np.polyval(F, -1.0), rtol=0,
                           atol=1e-12 * np.abs(ci).sum() * m)
    tt, P, Q, _ = mesh.section_tables(tau, n)
    assert np.array_equal(tt, tau)
    assert np.array_equal(P, np.hstack((np.zeros((n, 1)), np.eye(n)))) and np.array_equal(Q, np.eye(n))
    tt, P, Q, _ = mesh.section_tables(tau, n + 1)  # +1 is a test point and a support point
    assert np.array_equal(P[-1], np.eye(n + 1)[-1]) and np.array_equal(Q[-1], np.eye(n)[-1])


def test_grid_tables_layout():
    ps = PSparams([3, 2, 5])
    t = mesh.grid_tables(ps)
    assert list(t["m"]) == [4, 3, 6]
    sizes = [m * (1 + (n + 1) + n + m) for m, n in zip(t["m"], (3, 2, 5))]
    assert list(t["off"]) == [0, sizes[0], sizes[0] + sizes[1]] and t["pool"].size == sum(sizes)
    for i, n in enumerate((3, 2, 5)):
        want = mesh.section_tables(ps.tau(i), n + 1)
        for a, b in zip(mesh_oracle.unpack(t, i, n), want):
            assert np.array_equal(a, b)
    assert list(mesh.grid_tables(ps, m=2)["m"]) == [2, 2, 2]
    with pytest.raises(ValueError):
        mesh.grid_tables(ps, m=[3, 0, 3])


@pytest.mark.parametrize("variant,factor", VARIANTS)
def test_oracle_square_grid_is_the_integrated_defect(variant, factor):
    p, u, c, x0, O, _ = _setup(variant, factor)
    x = helpers.perturbed(x0)
    err = mesh_oracle.mesh_error(O, x, _square_grid(O.ps))
    g, _ = O.objfunc(helpers.copy_x(x))
    _check_square_grid(O, x, err, g)


@pytest.mark.parametrize("variant,factor", VARIANTS)
def test_emulator_equals_oracle_bit_for_bit(variant, factor):
    p, u, c, x0, O, P = _setup(variant, factor)
    E = MeshEmuEngine(P)
    xs = [x0, helpers.perturbed(x0)] + ([_solution(P)] if (variant, factor) == ("example", 1) else [])
    for tabs in (mesh.grid_tables(O.ps), _square_grid(O.ps)):
        E.set_mesh_grid(tabs)
        for x in xs:
            assert _same_bits(E.mesh_error(problem.xdict_to_vector(x)), mesh_oracle.mesh_error(O, x, tabs))


def _coast_state(O, x, i):
    """x with section i's states replaced by an rtol 1e-13 DOP853 integration of the oracle's vacuum dynamics from the
    section's first state (engine off, held attitude: only position and velocity move)."""
    from scipy.integrate import solve_ivp

    u, ut = O.u, O.u["t"]
    ua, ub, xa, xb, n = O.ps.get_index(i)
    to, tf = x["t"][i], x["t"][i + 1]
    X, _ = mesh_oracle.section_states(O, x, i)
    units = O._units3()

    def f(_, y):
        rh = O.dyn.dynamics_velocity_NoAir(X[0, 0:1], y[None, 0:3], X[0:1, 7:11], O._param(i), units)[0]
        return np.hstack((y[3:6] * u["velocity"] / u["position"], rh)) * (tf - to) * ut / 2.0

    s = np.hstack((-1.0, O.ps.tau(i)))
    sol = solve_ivp(f, (-1.0, 1.0), X[0, 1:7], method="DOP853", rtol=1e-13, atol=1e-15, t_eval=s)
    y = {k: np.array(v, copy=True) for k, v in x.items()}
    for r in range(n + 1):
        y["mass"][xa + r] = X[0, 0]
        y["position"][3 * (xa + r):3 * (xa + r) + 3] = sol.y[0:3, r]
        y["velocity"][3 * (xa + r):3 * (xa + r) + 3] = sol.y[3:6, r]
        y["quaternion"][4 * (xa + r):4 * (xa + r) + 4] = X[0, 7:11]
    return y


# Largest component estimate for n = 2 .. 7 (DESIGN.md section 11):
#   SECO  1.02e-06  8.53e-10  3.73e-12  2.05e-15  3.41e-16  3.32e-16
#   SEP2  1.01e-09  8.57e-14  2.27e-16  5.52e-16  2.27e-16  4.53e-16


@pytest.mark.parametrize("event", ["SECO", "SEP2"])
def test_vacuum_coast_estimate_falls_with_n(event):
    Lg = leaves.get("gmath")
    x_sol = _solution(helpers.compiled_plan(*helpers.example_problem(coord=Lg.coordinate_c)[:3], coord=Lg.coordinate_c))
    errs = []
    for n in range(2, 8):
        def mutate(inp, n=n):
            for e in inp["events"]:
                if e["name"] == event:
                    e["num_nodes"] = n

        p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c, mutate=mutate)
        i = p["event_index"][event]
        O = helpers.oracle_nlp(p, u, c, "gmath", "seqfma")
        ps0 = helpers.example_problem(coord=Lg.coordinate_c)[0]["ps_params"]
        x = _coast_state(O, mesh.transfer(x_sol, ps0, O.ps), i)
        errs.append(float(mesh_oracle.mesh_error(O, x, mesh.grid_tables(O.ps))[i].max()))
    floor = 1e-12
    for a, b in zip(errs, errs[1:]):
        assert b < a or max(a, b) < floor, errs
    assert errs[0] > 100 * errs[-1] and errs[-1] < 1e-9, errs


def _events():
    return helpers.example_inputs()["events"]


def test_refine_nodes_rule_cap_and_untouched_events():
    ev = _events()
    S = len(ev) - 1
    err = np.zeros((S, 11))
    err[0, 3] = 1e-3  # LIFTOFF, n = 5: 5 + ceil(log(1e4) / log(5)) = 11
    err[2, 5] = 2e-7  # ZEROLIFT_START, n = 16 > n_max: not split, reported
    err[3, 0] = 1e-1  # ZEROLIFT_END, n = 8: 8 + ceil(log(1e6) / log(8)) = 15, capped at 12
    err[4, 1] = 1e-7  # MECO: equal to tol, untouched
    err[6, 2] = 2e-7  # SEIG, n = 5: just above tol, + 1
    err[7, 9] = 1e2   # FAIRING, n = 6: 6 + 12, capped at 12
    new, rep = mesh.refine_nodes(ev, err, tol=1e-7, n_max=12)
    assert [r.name for r in rep] == [e["name"] for e in ev[:S]]
    got = {r.name: (r.n_old, r.n_new, r.capped) for r in rep}
    assert got["LIFTOFF"] == (5, 11, False)
    assert got["ZEROLIFT_START"] == (16, 16, True)
    assert got["ZEROLIFT_END"] == (8, 12, True)
    assert got["MECO"] == (2, 2, False)
    assert got["SEIG"] == (5, 6, False)
    assert got["FAIRING"] == (6, 12, True)
    assert all(r.n_new == r.n_old and not r.capped for r in rep if r.err == 0.0)
    assert rep[0].err == 1e-3
    for i, (a, b) in enumerate(zip(new, ev)):
        a, b = dict(a), dict(b)
        if i < S:
            assert a.pop("num_nodes") == rep[i].n_new
            b.pop("num_nodes")
        assert a.keys() == b.keys() and all(a[k] == b[k] or (a[k] != a[k] and b[k] != b[k]) for k in a)
    assert [e["num_nodes"] for e in ev] == [e["num_nodes"] for e in _events()]  # the input is not modified
    # the dictionary form of GelatoProblem.mesh_error; a non-finite estimate is refused
    new2, rep2 = mesh.refine_nodes(ev, {e["name"]: np.full(11, 1e-3) for e in ev[:S]}, tol=1e-6, n_max=40)
    assert [r.n_new for r in rep2] == [n + max(1, int(np.ceil(np.log(1e3) / np.log(max(n, 2))))) for n in
                                       (e["num_nodes"] for e in ev[:S])]
    with pytest.raises(ValueError):
        mesh.refine_nodes(ev, np.full((S, 11), np.nan), tol=1e-6, n_max=16)


def test_transfer_polynomials_identity_and_refined_plan():
    ps, ps2 = PSparams([3, 4, 2]), PSparams([3, 7, 5])
    rng = np.random.default_rng(3)
    M, N = ps.num_x(), ps.num_u()
    x = {"mass": np.empty(M), "position": np.empty(3 * M), "velocity": np.empty(3 * M), "quaternion": np.empty(4 * M),
         "u": np.empty(2 * N), "t": np.array([0.0, 0.1, 0.3, 0.5])}
    coef = {}
    for i in range(3):
        ua, ub, xa, xb, n = ps.get_index(i)
        s = np.hstack((-1.0, ps.tau(i)))
        for k, w in (("mass", 1), ("position", 3), ("velocity", 3), ("quaternion", 4)):
            c = rng.normal(size=(w, n + 1))
            coef[i, k] = c
            x[k].reshape(-1, w)[xa:xb] = np.stack([np.polyval(c[j], s) for j in range(w)], axis=1)
        c = rng.normal(size=(2, n))
        coef[i, "u"] = c
        x["u"].reshape(-1, 2)[ua:ub] = np.stack([np.polyval(c[j], ps.tau(i)) for j in range(2)], axis=1)
    y = mesh.transfer(x, ps, ps2)
    assert list(y) == list(x) and _same_bits(y["t"], x["t"])
    for i in range(3):
        ua, ub, xa, xb, n = ps2.get_index(i)
        s = np.hstack((-1.0, ps2.tau(i)))
        for k, w in (("mass", 1), ("position", 3), ("velocity", 3), ("quaternion", 4)):
            want = np.stack([np.polyval(coef[i, k][j], s) for j in range(w)], axis=1)
            assert np.allclose(y[k].reshape(-1, w)[xa:xb], want, rtol=0, atol=1e-12 * np.abs(coef[i, k]).sum())
        want = np.stack([np.polyval(coef[i, "u"][j], ps2.tau(i)) for j in range(2)], axis=1)
        assert np.allclose(y["u"].reshape(-1, 2)[ua:ub], want, rtol=0, atol=1e-12 * np.abs(coef[i, "u"]).sum())
        if i == 0:  # unrefined: bit for bit
            xa0, xb0 = ps.get_index(0)[2:4]
            assert _same_bits(y["position"].reshape(-1, 3)[xa:xb], x["position"].reshape(-1, 3)[xa0:xb0])
    same = mesh.transfer(x, ps, ps)
    assert all(_same_bits(same[k], x[k]) for k in x)
    # the example refined at tol 1e-6: the new plan builds and evaluates at the transferred solution
    Lg = leaves.get("gmath")
    p, u, c, _ = helpers.example_problem(coord=Lg.coordinate_c)
    P = helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c)
    x_sol = _solution(P)
    O = helpers.oracle_nlp(p, u, c, "gmath", "seqfma")
    err = mesh_oracle.mesh_error(O, x_sol, mesh.grid_tables(O.ps))
    inp = helpers.example_inputs()
    inp["events"], rep = mesh.refine_nodes(inp["events"], err, tol=1e-6, n_max=30)
    assert any(r.n_new > r.n_old for r in rep)
    p2, u2, c2, _ = problem.problem_from_inputs(inp, coord=Lg.coordinate_c)
    x2 = mesh.transfer(x_sol, p["ps_params"], p2["ps_params"])
    P2 = helpers.compiled_plan(p2, u2, c2, coord=Lg.coordinate_c)
    E = MeshEmuEngine(P2)
    g = E.eval_residuals(problem.xdict_to_vector(x2))
    assert g.shape == (P2.n_rows,) and np.isfinite(g).all()
    O2 = helpers.oracle_nlp(p2, u2, c2, "gmath", "seqfma")
    E.set_mesh_grid(mesh.grid_tables(O2.ps))
    err2 = E.mesh_error(problem.xdict_to_vector(x2))
    assert _same_bits(err2, mesh_oracle.mesh_error(O2, x2, mesh.grid_tables(O2.ps)))


def test_gelato_problem_mesh_error_on_the_emulator():
    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    prob = callbacks.GelatoProblem(p, u, c, user_eq=callbacks.PerigeeAtEvent(helpers.USER_EVENT), coord=Lg.coordinate_c,
                                   engine_factory=MeshEmuEngine)
    x = helpers.perturbed(x0)
    got = prob.mesh_error(x)
    want = mesh_oracle.mesh_error(helpers.oracle_nlp(p, u, c, "gmath", "seqfma"), x, mesh.grid_tables(p["ps_params"]))
    names = [e["name"] for e in p["params"][:-1]]
    assert list(got) == names
    assert _same_bits(np.stack([got[k] for k in names]), want)
    assert _same_bits(np.stack(list(prob.mesh_error(x).values())), want)  # the grid is set once, the result repeats
    prob.close()


# ------------------------------------------------------------------------------------------------ GPU tier
def _engine(P, scenario_plans=None):
    return engine.Engine(P, device=0, scenario_plans=scenario_plans)


@pytest.mark.gpu
@pytest.mark.parametrize("variant,factor", VARIANTS)
def test_gpu_equals_oracle_bit_for_bit(variant, factor):
    p, u, c, x0, O, P = _setup(variant, factor)
    E = _engine(P)
    xs = [x0, helpers.perturbed(x0)] + ([_solution(P)] if (variant, factor) == ("example", 1) else [])
    for tabs in (mesh.grid_tables(O.ps), _square_grid(O.ps)):
        E.set_mesh_grid(tabs)
        for x in xs:
            assert _same_bits(E.mesh_error(problem.xdict_to_vector(x)), mesh_oracle.mesh_error(O, x, tabs))
    E.close()


@pytest.mark.gpu
def test_gpu_square_grid_is_the_integrated_gpu_defect():
    p, u, c, x0, O, P = _setup("example", 3)
    E = _engine(P)
    x = helpers.perturbed(x0)
    E.set_mesh_grid(_square_grid(O.ps))
    err = E.mesh_error(problem.xdict_to_vector(x))
    g = P.split_residuals(E.eval_residuals(problem.xdict_to_vector(x)))
    _check_square_grid(O, x, err, g)
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
    X = np.stack([problem.xdict_to_vector(x) for x in xs])
    err = E.mesh_error(X, n_scen=64)
    for k in range(64):
        assert _same_bits(err[k], mesh_oracle.mesh_error(oracles[k], xs[k], tabs)), k
    # different scenarios give different estimates: the per-scenario blocks are read
    assert not _same_bits(err[0], err[1])
    E.close()


@pytest.mark.gpu
def test_gpu_bench_workload_sample():
    import bench

    Lg = leaves.get("gmath")
    plans, X, probs = bench.load_workload("example", 15, 128, 0, 128, coord=Lg.coordinate_c)
    E = _engine(plans[0], scenario_plans=plans)
    tabs = mesh.grid_tables(plans[0].ps)
    E.set_mesh_grid(tabs)
    err = E.mesh_error(X, n_scen=128)
    assert err.shape == (128, plans[0].S, 11) and np.isfinite(err).all()
    for k in (0, 37, 127):
        p, u, c, x = probs[k]
        assert _same_bits(err[k], mesh_oracle.mesh_error(helpers.oracle_nlp(p, u, c, "gmath", "seqfma"), x, tabs)), k
    E.close()


@pytest.mark.gpu
def test_gpu_host_dev_pinned_pageable_agree():
    import torch

    p, u, c, x0, O, P = _setup("example", 2)
    plans = [P] * 3
    E = _engine(P, scenario_plans=plans)
    E.set_mesh_grid(mesh.grid_tables(O.ps))
    X = np.stack([problem.xdict_to_vector(helpers.perturbed(x0, seed=k)) for k in range(3)])
    ref = E.mesh_error(X, n_scen=3)
    px, pe = engine.PinnedArray(X.size), engine.PinnedArray(ref.size)
    px.array[:] = X.ravel()
    E.mesh_error(px.array, n_scen=3, out=pe.array)
    assert _same_bits(pe.array.reshape(ref.shape), ref)
    xd = torch.from_numpy(X).cuda()
    ed = torch.full(ref.shape, float("nan"), dtype=torch.float64, device="cuda")
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        E.mesh_error_dev(xd.data_ptr(), ed.data_ptr(), 3, st.cuda_stream)
    st.synchronize()
    assert _same_bits(ed.cpu().numpy(), ref)
    assert _same_bits(E.mesh_error(X[1]), ref[1])  # a smaller batch after a larger one
    px.free()
    pe.free()
    E.close()


@pytest.mark.gpu
def test_gpu_argument_errors_leave_the_plan_usable_and_fd_mode_is_irrelevant():
    p, u, c, x0, O, P = _setup("example", 1)
    E = _engine(P)
    x = problem.xdict_to_vector(helpers.perturbed(x0))
    with pytest.raises(engine.GelatoError, match="no mesh grid"):
        E.mesh_error(x)
    tabs = mesh.grid_tables(O.ps)
    E.set_mesh_grid(tabs)
    ref = E.mesh_error(x)
    bad = []
    t = {k: v.copy() for k, v in tabs.items()}
    t["m"][3] = 0
    bad.append(t)
    t = {k: v.copy() for k, v in tabs.items()}
    t["off"][-1] = tabs["pool"].size - 1
    bad.append(t)
    t = {k: v.copy() for k, v in tabs.items()}
    t["off"][0] = -1
    bad.append(t)
    t = {k: v.copy() for k, v in tabs.items()}
    t["pool"][7] = np.nan
    bad.append(t)
    t = {k: v.copy() for k, v in tabs.items()}
    t["pool"][-1] = np.inf
    bad.append(t)
    t = {k: v.copy() for k, v in tabs.items()}
    t["m"][0] = 2 ** 31 - 1
    bad.append(t)
    for t in bad:
        with pytest.raises(engine.GelatoError, match="gelato_plan_set_mesh_grid"):
            E.set_mesh_grid(t)
        assert _same_bits(E.mesh_error(x), ref)
    L = E.L
    err = np.empty(P.S * 11)
    xp = x.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    ep = err.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    assert L.gelato_eval_mesh_error(E.h, xp, ep, 0) == -1
    assert L.gelato_eval_mesh_error(E.h, None, ep, 1) == -1
    assert L.gelato_plan_set_mesh_grid(E.h, None) == -1
    assert _same_bits(E.mesh_error(x), ref)
    E.set_fd("central")
    E.eval_jacobian(x)
    assert _same_bits(E.mesh_error(x), ref)
    E.close()
    # per-scenario blocks: an n_scen beyond the configured scenarios is refused
    E2 = _engine(P, scenario_plans=[P, P])
    E2.set_mesh_grid(tabs)
    with pytest.raises(engine.GelatoError, match="configured"):
        E2.mesh_error(np.stack([x] * 3), n_scen=3)
    assert _same_bits(E2.mesh_error(np.stack([x] * 2), n_scen=2)[1], ref)
    E2.close()
