"""Central-difference Jacobian mode (DESIGN.md H6): every finite-difference value is (q(+h) + q(-h)) * 0.5, q(+-h) being
the forward protocol (H3) run with step +-h; analytic and constant slots, sparsity, COO order, the packed layout and
objfunc do not change.

CPU tier: the oracle against the 4th-order derivative (closer than forward mode on every finite-difference block), the
kernels' code in the host emulator against the oracle bit for bit (signed zeros included: bit patterns are compared,
not values), GelatoProblem on the emulator, and the shared-reciprocal division with the negative divisor of the -h
pass.  GPU tier: the C ABI, through every entry point that returns Jacobian values, against the oracle."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import helpers
from central_oracle import CentralOracleNLP, Step, fd_quotient
from emu_central import FdEmuEngine
from gelato_b200 import callbacks, engine, problem, scenarios
from oracle import leaves, user_builtin

H = engine.DEFAULT_FD_STEP
HERE = os.path.dirname(os.path.abspath(__file__))

# Blocks of the example whose values depend on the step (profiles/r03a_fd_step_sweep.txt); every other block is
# analytic or constant and must keep forward mode's bits.
FD_BLOCKS = {
    "eqcon_dyn_quat/quaternion", "eqcon_dyn_quat/u", "eqcon_dyn_vel/mass", "eqcon_dyn_vel/position",
    "eqcon_dyn_vel/quaternion", "eqcon_dyn_vel/t", "eqcon_dyn_vel/velocity", "eqcon_pos/position", "eqcon_pos/t",
    "eqcon_terminal/position", "eqcon_terminal/velocity", "ineqcon_alpha/position", "ineqcon_alpha/quaternion",
    "ineqcon_alpha/t", "ineqcon_alpha/velocity", "ineqcon_antenna/position", "ineqcon_antenna/t", "ineqcon_iip/position",
    "ineqcon_iip/t", "ineqcon_iip/velocity", "ineqcon_qalpha/position", "ineqcon_qalpha/quaternion", "ineqcon_qalpha/t",
    "ineqcon_qalpha/velocity", "eqcon_user/mass", "eqcon_user/position", "eqcon_user/velocity", "eqcon_user/quaternion",
    "eqcon_user/u", "eqcon_user/t",
}
# Blocks whose rms error drops 100x or more at h = 1e-6 in that sweep: they must stay at least 10x closer.
DROP_100X = {
    "eqcon_dyn_quat/u", "eqcon_dyn_vel/mass", "eqcon_dyn_vel/quaternion", "eqcon_pos/position", "eqcon_terminal/position",
    "eqcon_terminal/velocity", "ineqcon_alpha/position", "ineqcon_alpha/quaternion", "ineqcon_alpha/t",
    "ineqcon_alpha/velocity", "ineqcon_antenna/position", "ineqcon_antenna/t", "ineqcon_iip/position", "ineqcon_iip/t",
    "ineqcon_iip/velocity", "ineqcon_qalpha/t",
}


def _bits(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64)).view(np.int64)


def assert_bits_equal(a, b, what=""):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    same = _bits(a) == _bits(b)
    assert same.all(), (what, int((~same).sum()), a[~same][:3], b[~same][:3])


def assert_sens_bits(sa, sb):
    """Bit-pattern comparison of two funcsSens dicts: groups, variable blocks, sparsity and every value."""
    fa, fb = helpers.flatten_sens(sa), helpers.flatten_sens(sb)
    assert list(fa) == list(fb)
    for k in fa:
        ra, ca, da, sha = fa[k]
        rb, cb, db, shb = fb[k]
        assert tuple(sha) == tuple(shb), k
        if ra is not None:
            assert np.array_equal(ra, rb) and np.array_equal(ca, cb), k
        assert_bits_equal(da, db, k)


def _oracle(p, u, c, derivative="central", fd_step=H, user=True, ue=None, ui=None):
    Lg = leaves.get("gmath")
    if user and ue is None:
        ue = user_builtin.perigee_ratio_at(Lg, helpers.USER_EVENT)
    return CentralOracleNLP(p, u, c, "gmath", "seqfma", user_eq=ue, user_ineq=ui, derivative=derivative, fd_step=fd_step)


def _setup(variant, factor=1, user=True, max_nodes=12):
    Lg = leaves.get("gmath")
    p, u, c, x0 = problem.problem_from_inputs(helpers.variant_inputs(variant), coord=Lg.coordinate_c, factor=factor,
                                              max_nodes=max_nodes)
    return p, u, c, x0, _oracle(p, u, c, user=user), helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c, user=user)


def _user_setup():
    Lg = leaves.get("gmath")
    eq_rows = [("orbit_energy", -3.0e7, 1.0)]
    ineq_rows = [("eccentricity", 0.05, 0.5), ("semi_major_axis", 6578137.0, 1.0)]
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c, factor=2, max_nodes=12)
    O = _oracle(p, u, c, ue=user_builtin.orbit_rows_at(Lg, helpers.USER_EVENT, eq_rows),
                ui=user_builtin.orbit_rows_at(Lg, "SECO", ineq_rows))
    from gelato_b200 import plan as gplan

    P = gplan.CompiledPlan(p, u, c, user_eq=gplan.OrbitAtEvent(helpers.USER_EVENT, eq_rows),
                           user_ineq=gplan.OrbitAtEvent("SECO", ineq_rows), coord=Lg.coordinate_c)
    return p, u, c, x0, O, P


VARIANTS = [("example", 1, True), ("example", 3, True), ("fuel_inclination", 1, True), ("all_aero", 2, True),
            ("waypoints", 1, True), ("neg_area", 1, True), ("three_stage", 1, True), ("iip_orbital", 1, True),
            ("bare", 1, False), ("user_registry", 2, True)]


def _case(variant, factor, user):
    if variant == "user_registry":
        return _user_setup()
    return _setup(variant, factor, user)


# ------------------------------------------------------------------------------------------------ CPU tier
def test_oracle_central_is_closer_to_the_derivative_and_leaves_the_rest_alone():
    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    x = helpers.perturbed(x0)
    F, C = _oracle(p, u, c, "forward"), _oracle(p, u, c)
    row0, J, col0 = helpers.true_jacobian(F.objfunc, x)
    sf, _ = F.sens(helpers.copy_x(x))
    xc = helpers.copy_x(x)
    sc, _ = C.sens(xc)
    assert all(np.array_equal(_bits(xc[k]), _bits(x[k])) for k in x), "central sens perturbs copies only"
    ef, ec = helpers.derivative_errors(sf, row0, J, col0), helpers.derivative_errors(sc, row0, J, col0)
    ff, fc = helpers.flatten_sens(sf), helpers.flatten_sens(sc)
    assert list(ff) == list(fc)
    moved = set()
    for k in ff:
        assert tuple(ff[k][3]) == tuple(fc[k][3]), k
        if ff[k][0] is not None:
            assert np.array_equal(ff[k][0], fc[k][0]) and np.array_equal(ff[k][1], fc[k][1]), k
        if not np.array_equal(_bits(ff[k][2]), _bits(fc[k][2])):
            moved.add(k)
    assert moved <= FD_BLOCKS, moved - FD_BLOCKS  # analytic and constant blocks: forward mode's bits
    rms = lambda a: float(np.sqrt(np.mean(np.square(a))))  # noqa: E731
    for k in sorted(moved & set(ef)):
        assert ec[k].max() <= ef[k].max() and rms(ec[k]) <= rms(ef[k]), (k, ec[k].max(), ef[k].max())
    for k in DROP_100X:
        assert rms(ec[k]) * 10.0 <= rms(ef[k]), (k, rms(ec[k]), rms(ef[k]))
    fa, _ = F.objfunc(helpers.copy_x(x))
    fb, _ = C.objfunc(helpers.copy_x(x))
    for k in fa:
        if fa[k] is not None:
            assert_bits_equal(fa[k], fb[k], k)


def test_oracle_central_is_the_mean_of_the_two_forward_passes():
    p, u, c, x0 = helpers.example_problem()
    x = helpers.perturbed(x0)
    C = _oracle(p, u, c, fd_step=3e-7)
    F = _oracle(p, u, c, "forward")
    F.dx = Step(3e-7)
    sp, _ = F.sens(helpers.copy_x(x))
    F.dx = Step(-3e-7)
    sm, _ = F.sens(helpers.copy_x(x))
    sc, _ = C.sens(helpers.copy_x(x))
    for k, (_, _, d, _) in helpers.flatten_sens(sc).items():
        assert_bits_equal(d, (helpers.flatten_sens(sp)[k][2] + helpers.flatten_sens(sm)[k][2]) * 0.5, k)


def test_zero_quotient_keeps_the_numerator_sign():
    """The kernels' rule for a zero numerator (jobs.h: fd_div), which the oracle follows: the zero comes back as it
    is, so the -h pass does not flip the sign IEEE's 0 / (-h) would."""
    num = np.array([0.0, -0.0, 1e-20, -3.0])
    for dx in (1e-8, -1e-6):
        q = fd_quotient(num, dx)
        assert_bits_equal(q[:2], num[:2])
        assert_bits_equal(q[2:], num[2:] / dx)


@pytest.mark.parametrize("variant,factor,user", VARIANTS)
def test_emulated_central_matches_oracle_bitwise(variant, factor, user):
    p, u, c, x0, O, P = _case(variant, factor, user)
    E = FdEmuEngine(P)
    E.set_fd("central", H)
    F = FdEmuEngine(P)
    full, src, sgn = E.packed_map()
    for x in (x0, helpers.perturbed(x0)):
        xv = problem.xdict_to_vector(x)
        order = list(x.keys())
        s, _ = O.sens(helpers.copy_x(x))
        vals = E.eval_jacobian(xv)
        assert not np.isnan(vals).any()
        assert_sens_bits(s, P.split_jacobian(vals, key_order=order))
        # pair, COO: the same values, g = objfunc's rows
        g_want = F.eval_residuals(xv)
        g, v = E.eval_pair(xv)
        assert_bits_equal(v, vals, "pair vals")
        assert_bits_equal(g, g_want, "pair g")
        # packed, sens only and pair: template + map(packed) = the COO values
        for pk in (E.eval_jacobian_packed(xv), E.eval_pair(xv, packed=True)[1]):
            v2 = P.vals_template.copy()
            v2[full] = sgn * pk[src]
            assert_bits_equal(v2, vals, "packed")
        assert_bits_equal(E.eval_pair(xv, packed=True)[0], g_want, "packed pair g")


def test_emulated_central_dispersed_scenarios_with_ids():
    Lg = leaves.get("gmath")
    scen = scenarios.disperse(helpers.example_inputs(), 3, seed=20260117)
    plans, oracles, xs = [], [], []
    for si in scen:
        p, u, c, x0 = problem.problem_from_inputs(si, coord=Lg.coordinate_c)
        plans.append(helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c))
        oracles.append(_oracle(p, u, c))
        xs.append(helpers.perturbed(x0, seed=len(xs)))
    E = FdEmuEngine(plans[0], scenario_plans=plans)
    E.set_fd("central")
    ids = [2, 0, 2, 1]
    X = np.stack([problem.xdict_to_vector(xs[i]) for i in ids])
    V = E.eval_jacobian(X, n_scen=4, scen_ids=ids)
    G, PK = E.eval_pair(X, n_scen=4, scen_ids=ids, packed=True)
    full, src, sgn = E.packed_map()
    for k, i in enumerate(ids):
        s, _ = oracles[i].sens(helpers.copy_x(xs[i]))
        assert_sens_bits(s, plans[i].split_jacobian(V[k], key_order=list(xs[i].keys())))
        v2 = plans[i].vals_template.copy()
        v2[full] = sgn * PK[k][src]
        assert_bits_equal(v2, V[k])
    assert not np.array_equal(V[0], V[3])


def _problem_on_emulator(derivative="forward", fd_step=None, **kw):
    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    prob = callbacks.GelatoProblem(p, u, c, user_eq=callbacks.PerigeeAtEvent(helpers.USER_EVENT), coord=Lg.coordinate_c,
                                   engine_factory=FdEmuEngine, derivative=derivative, fd_step=fd_step, **kw)
    return prob, p, u, c, x0


@pytest.mark.parametrize("kw", [{}, {"reuse_output": False}, {"fuse_pair": True}])
def test_gelato_problem_central_on_the_emulator(kw):
    prob, p, u, c, x0 = _problem_on_emulator("central", **kw)
    assert prob.engine.fd == ("central", H)
    ref, _, _, _, _ = _problem_on_emulator()
    O = _oracle(p, u, c)
    for seed in (1, 2):
        x = helpers.perturbed(x0, seed=seed)
        f, _ = prob.objfunc(x)
        helpers.assert_funcs_equal(f, ref.objfunc(x)[0])
        s, _ = prob.sens(x, f)
        assert_sens_bits(O.sens(helpers.copy_x(x))[0], s)
    # jacobian_csr follows the mode too
    x = helpers.perturbed(x0, seed=3)
    csr = prob.jacobian_csr(x)
    vals = FdEmuEngine(prob.plan)
    vals.set_fd("central")
    m = prob.plan.csr_map(key_order=tuple(x.keys()))
    assert_bits_equal(csr.data, np.append(vals.eval_jacobian(problem.xdict_to_vector(x)), 0.0)[m["src"]])


def test_switching_back_to_forward_gives_the_bits_of_a_problem_never_switched():
    A, p, u, c, x0 = _problem_on_emulator()
    B, _, _, _, _ = _problem_on_emulator("central", fd_step=3e-7)
    x = helpers.perturbed(x0)
    sa = A.sens(x)[0]
    sa = helpers.flatten_sens(sa)
    sa = {k: (v[0], v[1], np.array(v[2]), v[3]) for k, v in sa.items()}  # copies: the views move with the buffer
    B.sens(x)
    B.engine.set_fd("forward")
    assert B.engine.fd == ("forward", float(p["dx"]))
    sb = helpers.flatten_sens(B.sens(x)[0])
    for k in sa:
        assert_bits_equal(sa[k][2], sb[k][2], k)


@pytest.mark.parametrize("bad", [dict(derivative="backward"), dict(derivative="central", fd_step=0.0),
                                 dict(derivative="central", fd_step=-1e-6), dict(derivative="central", fd_step=2e-3),
                                 dict(derivative="central", fd_step=float("nan")),
                                 dict(derivative="central", fd_step=float("inf")), dict(derivative="central", fd_step="1e-6")])
def test_bad_derivative_arguments_are_rejected(bad):
    with pytest.raises(ValueError):
        _problem_on_emulator(**bad)
    prob, p, u, c, _ = _problem_on_emulator()
    with pytest.raises(ValueError):
        prob.engine.set_fd(bad["derivative"], bad.get("fd_step"))
    assert prob.engine.fd == ("forward", float(p["dx"]))
    with pytest.raises(ValueError):
        _oracle(p, u, c, bad["derivative"], bad.get("fd_step"))


def test_shared_reciprocal_division_with_negative_divisors():
    """gm_div_by(a, gm_rcp(-h)) -- the -h pass's quotients -- gives the bits of IEEE a / (-h), for the steps a user
    may set and numerators over the range of finite differences of the right-hand sides."""
    lib = os.path.join(HERE, "_build", "libgmath_shim_fd.so")
    os.makedirs(os.path.dirname(lib), exist_ok=True)
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-mfma", "-shared", "-fPIC", "-o", lib,
                           os.path.join(HERE, "gmath_host_shim.c"), "-lm"])
    shim = ctypes.CDLL(lib)
    pd = ctypes.POINTER(ctypes.c_double)
    rng = np.random.default_rng(17)
    steps = np.concatenate(([1e-3, 1e-6, 1e-7, 3e-7, 1e-8, 5e-324, 2.2250738585072014e-308], 10.0 ** rng.uniform(-12, -3, 2000)))
    n = 400
    a = np.concatenate((rng.standard_normal(steps.size * n) * 10.0 ** rng.uniform(-300, 10, steps.size * n),
                        np.tile([0.0, -0.0, 1.0, -1.0, np.inf, np.nan], steps.size)))
    d = -np.concatenate((np.repeat(steps, n), np.repeat(steps, 6)))
    got = np.empty_like(a)
    shim.gmt_div_by(a.ctypes.data_as(pd), d.ctypes.data_as(pd), got.ctypes.data_as(pd), a.size)
    with np.errstate(all="ignore"):
        want = a / d
    same = (_bits(got) == _bits(want)) | (np.isnan(got) & np.isnan(want))
    assert same.all(), (a[~same][:5], d[~same][:5])


# ------------------------------------------------------------------------------------------------ GPU tier
def _gpu_engine(P, scenario_plans=None):
    E = engine.Engine(P, scenario_plans=scenario_plans)
    E.set_fd("central", H)
    return E


@pytest.mark.gpu
@pytest.mark.parametrize("variant,factor,user", VARIANTS)
def test_capi_central_matches_oracle_bitwise(variant, factor, user):
    import torch

    p, u, c, x0, O, P = _case(variant, factor, user)
    E = _gpu_engine(P)
    Fwd = engine.Engine(P)
    full, src, sgn = E.packed_map()
    for x in (x0, helpers.perturbed(x0)):
        xv = problem.xdict_to_vector(x)
        s, _ = O.sens(helpers.copy_x(x))
        vals = E.eval_jacobian(xv).copy()
        assert_sens_bits(s, P.split_jacobian(vals, key_order=list(x.keys())))
        g_want = Fwd.eval_residuals(xv).copy()
        assert_bits_equal(E.eval_jacobian(xv, scen_ids=[0]), vals, "_ids")
        for zero_copy in (False, True):
            E.set_update_zero_copy(zero_copy)
            for pinned in (False, True):
                hv = engine.PinnedArray(P.n_vals) if pinned else None
                buf = hv.array if pinned else np.empty(P.n_vals)
                E.jacobian_template(buf, 1)
                assert_bits_equal(E.eval_jacobian_update(xv, buf, 1), vals, "_update")
                g = np.empty(P.n_rows)
                buf[P.xdep_index()] = np.nan
                G, V = E.eval_pair_update(xv, g, buf, 1)
                assert_bits_equal(V[0], vals, "pair_update")
                assert_bits_equal(G[0], g_want, "pair_update g")
                if hv is not None:
                    hv.free()
        v2 = P.vals_template.copy()
        v2[full] = sgn * E.eval_jacobian_packed(xv)[src]
        assert_bits_equal(v2, vals, "_packed")
        for g, pk in (E.eval_pair_packed(xv), E.eval_pair_packed(xv, scen_ids=[0])):
            v2[full] = sgn * pk[src]
            assert_bits_equal(v2, vals, "pair_packed")
            assert_bits_equal(g, g_want, "pair_packed g")
        # device-resident entry points
        xd = torch.from_numpy(xv).cuda()
        gd = torch.full((P.n_rows,), float("nan"), dtype=torch.float64, device="cuda")
        vd = torch.full((P.n_vals,), float("nan"), dtype=torch.float64, device="cuda")
        pd = torch.full((E.n_pack,), float("nan"), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        E.fill_template(vd.data_ptr(), 1)
        E.eval_jacobian_dev(xd.data_ptr(), vd.data_ptr(), 1)
        torch.cuda.synchronize()
        assert_bits_equal(vd.cpu().numpy(), vals, "_dev")
        vd.fill_(float("nan"))
        torch.cuda.synchronize()
        E.fill_template(vd.data_ptr(), 1)
        E.eval_pair_dev(xd.data_ptr(), gd.data_ptr(), vd.data_ptr(), 1)
        torch.cuda.synchronize()
        assert_bits_equal(vd.cpu().numpy(), vals, "pair_dev")
        assert_bits_equal(gd.cpu().numpy(), g_want, "pair_dev g")
        gd.fill_(float("nan"))
        torch.cuda.synchronize()
        E.eval_pair_packed_dev(xd.data_ptr(), gd.data_ptr(), pd.data_ptr(), 1)
        torch.cuda.synchronize()
        v2[full] = sgn * pd.cpu().numpy()[src]
        assert_bits_equal(v2, vals, "pair_packed_dev")
        assert_bits_equal(gd.cpu().numpy(), g_want, "pair_packed_dev g")
    E.close()
    Fwd.close()


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [True, False])
def test_capi_central_sliced_batches_of_dispersed_scenarios(pinned):
    """Update and packed mode cut a batch into slices on several streams, each with its own region of the scratch;
    subsets by scenario id.  Every scenario against its own oracle."""
    Lg = leaves.get("gmath")
    n = 7
    scen = scenarios.disperse(helpers.example_inputs(), n, seed=5)
    plans, oracles, xs = [], [], []
    for si in scen:
        p, u, c, x0 = problem.problem_from_inputs(si, coord=Lg.coordinate_c, factor=2)
        plans.append(helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c))
        oracles.append(_oracle(p, u, c))
        xs.append(helpers.perturbed(x0, seed=3 + len(xs)))
    P = plans[0]
    E = _gpu_engine(P, scenario_plans=plans)
    X = np.stack([problem.xdict_to_vector(x) for x in xs])
    V = E.eval_jacobian(X, n_scen=n).copy()
    for k in range(n):
        assert_sens_bits(oracles[k].sens(helpers.copy_x(xs[k]))[0], plans[k].split_jacobian(V[k], key_order=list(xs[k].keys())))
    g_want = engine.Engine(P, scenario_plans=plans).eval_residuals(X, n).copy()
    full, src, sgn = E.packed_map()
    hv = engine.PinnedArray(n * P.n_vals) if pinned else None
    v = hv.array if pinned else np.empty(n * P.n_vals)
    E.jacobian_template(v, n)
    for zero_copy in (False, True):
        E.set_update_zero_copy(zero_copy)
        for slices in (1, 3, 0):
            E.set_update_slices(slices)
            v.reshape(n, -1)[:, P.xdep_index()] = np.nan
            g = np.empty(n * P.n_rows)
            G, VV = E.eval_pair_update(X, g, v, n)
            assert_bits_equal(VV, V, (zero_copy, slices))
            assert_bits_equal(G, g_want, (zero_copy, slices))
            v.reshape(n, -1)[:, P.xdep_index()] = np.nan
            assert_bits_equal(E.eval_jacobian_update(X, v, n), V, (zero_copy, slices))
            G, PK = E.eval_pair_packed(X, n_scen=n)
            assert_bits_equal(G, g_want)
            for k in range(n):
                v2 = plans[k].vals_template.copy()
                v2[full] = sgn * PK[k][src]
                assert_bits_equal(v2, V[k])
    ids = [6, 0, 6, 3]
    assert_bits_equal(E.eval_jacobian(X[ids], n_scen=4, scen_ids=ids), V[ids])
    G, PK = E.eval_pair_packed(X[ids], n_scen=4, scen_ids=ids)
    assert_bits_equal(G, g_want[ids])
    if hv is not None:
        hv.free()
    E.close()


@pytest.mark.gpu
def test_capi_central_at_the_bench_workload_against_the_emulator():
    """The bench workload (example x15, N = 990): a few scenarios of a pair evaluation, bit for bit against the
    emulator; g equals the forward objfunc rows."""
    import torch

    p, u, c, x0 = helpers.example_problem(factor=15, max_nodes=20)
    P = helpers.compiled_plan(p, u, c)
    n = 3
    X = np.stack([problem.xdict_to_vector(helpers.perturbed(x0, seed=40 + k)) for k in range(n)])
    E = _gpu_engine(P)
    F = engine.Engine(P)
    xd = torch.from_numpy(X).cuda()
    gd = torch.full((n, P.n_rows), float("nan"), dtype=torch.float64, device="cuda")
    pd = torch.full((n, E.n_pack), float("nan"), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    E.eval_pair_packed_dev(xd.data_ptr(), gd.data_ptr(), pd.data_ptr(), n)
    torch.cuda.synchronize()
    Em = FdEmuEngine(P)
    Em.set_fd("central", H)
    g_emu, pk_emu = Em.eval_pair(X, n_scen=n, packed=True)
    assert_bits_equal(pd.cpu().numpy(), pk_emu)
    assert_bits_equal(gd.cpu().numpy(), g_emu)
    assert_bits_equal(gd.cpu().numpy(), F.eval_residuals(X, n))
    E.close()
    F.close()


@pytest.mark.gpu
def test_capi_mode_switches_errors_and_the_range_entry_point():
    import torch

    p, u, c, x0, O, P = _setup("example", 2)
    E, never = engine.Engine(P), engine.Engine(P)
    xv = problem.xdict_to_vector(helpers.perturbed(x0))
    want = never.eval_jacobian(xv).copy()
    dx = float(p["dx"])
    assert E.fd == ("forward", dx)
    E.set_fd("central", 2e-7)
    assert E.fd == ("central", 2e-7)
    central = E.eval_jacobian(xv).copy()
    assert not np.array_equal(central, want)
    # argument errors leave the plan as it was
    code = ctypes.c_int32
    for mode, step in ((2, 1e-6), (-1, 1e-6), (1, 0.0), (1, -1e-6), (1, 1.1e-3), (1, float("nan")), (1, float("inf"))):
        assert E.L.gelato_plan_set_fd(E.h, code(mode), ctypes.c_double(step)) == -1
        assert E.fd == ("central", 2e-7)
    assert_bits_equal(E.eval_jacobian(xv), central)
    # the range evaluation refuses central mode ...
    xd = torch.from_numpy(xv).cuda()
    gd = torch.zeros(P.n_rows, dtype=torch.float64, device="cuda")
    pd = torch.zeros(E.n_pack, dtype=torch.float64, device="cuda")
    with pytest.raises(engine.GelatoError):
        E.eval_pair_packed_range_dev(xd.data_ptr(), gd.data_ptr(), pd.data_ptr(), (0, E.n_jac_blocks_pair),
                                     (0, E.n_vacuum_nodes))
    # ... and forward again is the never-switched plan, bit for bit
    E.set_fd("forward")
    assert E.fd == ("forward", dx)
    assert_bits_equal(E.eval_jacobian(xv), want)
    E.eval_pair_packed_range_dev(xd.data_ptr(), gd.data_ptr(), pd.data_ptr(), (0, E.n_jac_blocks_pair), (0, E.n_vacuum_nodes))
    torch.cuda.synchronize()
    g, pk = never.eval_pair_packed(xv)
    assert_bits_equal(pd.cpu().numpy(), pk)
    assert_bits_equal(gd.cpu().numpy(), g)
    E.close()
    never.close()
