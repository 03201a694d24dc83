"""Result-table user constraints (gelato_b200.plan.TableAtEvent, include/gelato_b200.h: GT_*; DESIGN.md section 10
"a16"): any column of the reference's result table at a named event, with jac_fd's dense Jacobian.

The truth is the oracle: tests/table_oracle.py writes the function the way a user_constraints.py would (the event row of
xdict through the oracle's output_row), and the oracle's jac_fd runs over it.  CPU tier: the host emulator of the
kernels (tests/emu) against it, bit for bit (NaN where the oracle has NaN).  GPU tier (-m gpu): the CUDA engine
through every entry point that writes g or Jacobian values, against the emulator and the oracle.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import central_oracle
import emu_binding
import emu_table
import helpers
import table_oracle
from gelato_b200 import callbacks, engine, output, problem, scenarios
from gelato_b200 import plan as gplan
from oracle import leaves, nlp

HERE = os.path.dirname(os.path.abspath(__file__))
AIR_EVENT, VACUUM_EVENT = "KICKTURN", "SECO"
# every column once; scales and offsets of both signs, and the plain column (scale 1, offset 0)
ALL_ROWS = [(c, (1.0, -250.0, 3.5)[k % 3], (0.0, 0.25, -1.5)[k % 3]) for k, c in enumerate(output.KERNEL_COLUMNS)]


def _builtin(kind, ev, rows):
    return (gplan.OrbitAtEvent if kind == "orbit" else gplan.TableAtEvent)(ev, rows)


def _user(spec, Lg):
    """spec: None, one (kind, event, rows) or a list of them -> (the plan's built-in(s), the oracle's user function)."""
    if spec is None:
        return None, None
    if isinstance(spec, tuple):
        return _builtin(*spec), table_oracle.group_rows_at(Lg, [spec])
    return [_builtin(*s) for s in spec], table_oracle.group_rows_at(Lg, spec)


def _setup(eq, ineq=None, variant="example", factor=1, max_nodes=12, central=False, inp=None):
    Lg = leaves.get("gmath")
    inp = inp if inp is not None else helpers.variant_inputs(variant)
    p, u, c, x0 = problem.problem_from_inputs(inp, coord=Lg.coordinate_c, factor=factor, max_nodes=max_nodes)
    be, oe = _user(eq, Lg)
    bi, oi = _user(ineq, Lg)
    cls = central_oracle.CentralOracleNLP if central else nlp.OracleNLP
    kw = {"derivative": "central"} if central else {}
    O = cls(p, u, c, "gmath", "seqfma", user_eq=oe, user_ineq=oi, **kw)
    P = gplan.CompiledPlan(p, u, c, user_eq=be, user_ineq=bi, coord=Lg.coordinate_c)
    return p, u, c, x0, O, P


def _same(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def assert_funcs_same(fa, fb):
    assert list(fa) == list(fb)
    for k in fa:
        assert (fa[k] is None) == (fb[k] is None), k
        if fa[k] is not None:
            assert _same(np.atleast_1d(fa[k]), np.atleast_1d(fb[k])), k


def assert_sens_same(sa, sb):
    assert list(sa) == list(sb)
    for k in sa:
        assert (sa[k] is None) == (sb[k] is None), k
        if sa[k] is None:
            continue
        assert list(sa[k]) == list(sb[k]), k
        for var, a in sa[k].items():
            b = sb[k][var]
            if isinstance(a, dict):
                assert all(np.array_equal(a["coo"][i], b["coo"][i]) for i in range(2)), (k, var)
                assert _same(a["coo"][2], b["coo"][2]), (k, var)
            else:
                assert _same(a, b), (k, var, np.nanmax(np.abs(np.asarray(a) - np.asarray(b))))


def _check(O, P, E, xs):
    for x in xs:
        xv = problem.xdict_to_vector(x)
        with np.errstate(all="ignore"):
            f, _ = O.objfunc(helpers.copy_x(x))
            s, _ = O.sens(helpers.copy_x(x))
        assert_funcs_same(f, P.split_residuals(E.eval_residuals(xv)))
        assert_sens_same(s, P.split_jacobian(E.eval_jacobian(xv), key_order=list(x.keys())))


def _solution(p):
    rec = np.load(os.path.join(HERE, "golden", "example_solution.npz"))
    return problem.vector_to_xdict(rec["x"], p["M"], p["N"], p["num_sections"])


# ---------------------------------------------------------------------------------------------------- CPU tier
@pytest.mark.parametrize("central", [False, True])
@pytest.mark.parametrize("event", [AIR_EVENT, VACUUM_EVENT])
def test_every_column_matches_the_oracle(event, central):
    p, u, c, x0, O, P = _setup(("table", event, ALL_ROWS), max_nodes=20, central=central)
    E = emu_table.TableEmulator(P)
    if central:
        E.set_fd("central")
    _check(O, P, E, (x0, helpers.perturbed(x0), _solution(p)))


@pytest.mark.parametrize("event", ["LIFTOFF", "SEP2"])
def test_events_at_the_first_and_last_section(event):
    rows = [("altitude", 1000.0, 0.0), ("downrange", 1e4, 1.0), ("vel_ground_NED_Z", -3.0, 0.0), ("M", 1.0, 0.0)]
    p, u, c, x0, O, P = _setup(("table", event, rows), ineq=("table", event, rows[::-1]))
    assert P.tab_i32[0, gplan.GT_TIDX] == p["event_index"][event]
    _check(O, P, emu_table.TableEmulator(P), (x0, helpers.perturbed(x0)))


@pytest.mark.parametrize("variant", ["three_stage", "neg_area", "all_aero"])
def test_constraint_variants(variant):
    rows = [("dynamic_pressure", 1e4, 0.0), ("accel_BODY_X", 9.8, 1.0), ("aero_BODY_X", 1e3, 0.0), ("thrust", 1e5, 0.0)]
    p, u, c, x0, O, P = _setup(("table", "ZEROLIFT_START", rows), ineq=("table", VACUUM_EVENT, rows[:2]), variant=variant)
    _check(O, P, emu_table.TableEmulator(P), (x0, helpers.perturbed(x0)))


MIXED_EQ = [("orbit", "IIP_END", [("perigee_radius", 6378137.0, 1.0)]),
            ("table", "FAIRING", [("altitude", 1e5, 1.0), ("dynamic_pressure", 10.0, 0.0)])]
MIXED_INEQ = [("table", AIR_EVENT, [("AOA_total", 5.0, 0.0)]),
              ("table", VACUUM_EVENT, [("flightpath_vel_inertial_geocentric", 1.0, 0.0), ("altitude_perigee", 1e5, 1.0)])]


@pytest.mark.parametrize("central", [False, True])
@pytest.mark.parametrize("variant", ["example", "waypoints", "all_aero"])
def test_mixed_lists_and_the_residue_later_groups_see(variant, central):
    """A group of several built-ins is ONE jac_fd pass: each built-in's rows from its own read variables, one residue
    on every variable for the groups after it (aero, IIP, antenna rows: every group equals the oracle's)."""
    p, u, c, x0, O, P = _setup(MIXED_EQ, MIXED_INEQ, variant=variant, central=central)
    assert P.group_rows["eqcon_user"][1] == 3 and P.group_rows["ineqcon_user"][1] == 3 and P.n_tab == 3
    E = emu_table.TableEmulator(P)
    if central:
        E.set_fd("central")
    _check(O, P, E, (x0, helpers.perturbed(x0)))


def test_one_row_in_all_is_a_scalar_and_single_orbit_groups_keep_their_layout():
    p, u, c, x0, O, P = _setup(("table", AIR_EVENT, [("altitude", 1e3, 0.0)]))
    f, _ = O.objfunc(helpers.copy_x(x0))
    assert np.ndim(f["eqcon_user"]) == 0
    assert np.ndim(P.split_residuals(emu_table.TableEmulator(P).eval_residuals(problem.xdict_to_vector(x0)))["eqcon_user"]) == 0
    Lg = leaves.get("gmath")
    a = gplan.CompiledPlan(p, u, c, user_eq=gplan.PerigeeAtEvent("IIP_END"), coord=Lg.coordinate_c)
    b = gplan.CompiledPlan(p, u, c, user_eq=[gplan.PerigeeAtEvent("IIP_END")], coord=Lg.coordinate_c)
    assert a.n_tab == 0 and a.n_vals == b.n_vals and a.eval_counts() == b.eval_counts()
    for name in ("evt_i32", "evt_i64", "evt_f64", "vals_template", "rc_aero"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), name


def test_pair_packed_outputs_and_csr():
    p, u, c, x0, O, P = _setup(MIXED_EQ, MIXED_INEQ)
    E = emu_table.TableEmulator(P)
    full, src, sgn = E.packed_map()
    assert np.array_equal(full, P.xdep_index())
    for x in (x0, helpers.perturbed(x0)):
        xv = problem.xdict_to_vector(x)
        g_ref, v_ref = E.eval_residuals(xv), E.eval_jacobian(xv)
        g, v = E.eval_pair(xv)
        assert _same(g, g_ref) and _same(v, v_ref)
        g, pk = E.eval_pair(xv, packed=True)
        v = P.vals_template.copy()
        v[full] = sgn * pk[src]
        assert _same(g, g_ref) and _same(v, v_ref)
    prob = callbacks.GelatoProblem(p, u, c, user_eq=[_builtin(*s) for s in MIXED_EQ],
                                   user_ineq=[_builtin(*s) for s in MIXED_INEQ], coord=leaves.get("gmath").coordinate_c,
                                   engine_factory=emu_table.TableEmuEngine)
    x = helpers.perturbed(x0, seed=3)
    J = prob.jacobian_csr(x).toarray()
    so, _ = O.sens(helpers.copy_x(x))
    want = np.zeros_like(J)
    col0 = dict(zip(gplan.VAR_ORDER, np.cumsum([0] + [P.sizes[k] for k in gplan.VAR_ORDER])[:-1]))
    r0 = 0
    for key in gplan.GROUPS:
        if so.get(key) is None:
            continue
        nrow = P.group_rows[key][1]
        for var, blk in so[key].items():
            if isinstance(blk, dict):
                r, cc, d = blk["coo"]
                want[r0 + np.asarray(r), col0[var] + np.asarray(cc)] = d
            else:
                want[r0: r0 + nrow, col0[var]: col0[var] + P.sizes[var]] = np.reshape(blk, (nrow, -1))
        r0 += nrow
    assert _same(J, want)
    # the dense blocks of later sens calls are refreshed in place (update mode's dictionary)
    s1, _ = prob.sens(helpers.copy_x(x))
    s2, _ = prob.sens(helpers.copy_x(x0))
    so2, _ = O.sens(helpers.copy_x(x0))
    assert_sens_same(so2, s2)
    prob.close()


def _omega_cross_r(x, P, row):
    pos = x["position"][3 * row: 3 * row + 3] * P.u["position"]
    w = 7.2921151467e-5
    x["velocity"][3 * row: 3 * row + 3] = np.array([-w * pos[1], w * pos[0], 0.0]) / P.u["velocity"]


@pytest.mark.parametrize("case", ["no_impact_point", "zero_air_speed"])
def test_edge_states(case):
    """No impact point (orbital speed: lat_IIP / lon_IIP are NaN, fill_na = False) and zero air-relative velocity
    (Mach 0, the angles of attack of a zero vector): equal bits, NaN in the same places."""
    event = VACUUM_EVENT if case == "no_impact_point" else "LIFTOFF"
    p, u, c, x0, O, P = _setup(("table", event, ALL_ROWS), central=False)
    x = helpers.copy_x(x0)
    if case == "zero_air_speed":
        _omega_cross_r(x, P, int(P.tab_i32[0, gplan.GT_SROW]))
    E = emu_table.TableEmulator(P)
    g = P.split_residuals(E.eval_residuals(problem.xdict_to_vector(x)))["eqcon_user"]
    k = output.KERNEL_COLUMNS.index
    if case == "no_impact_point":
        assert np.isnan(g[[k("lat_IIP"), k("lon_IIP")]]).all()
    else:
        assert g[k("M")] == 0.0 and g[k("vel_air")] == 0.0
    _check(O, P, E, (x,))
    C = central_oracle.CentralOracleNLP(p, u, c, "gmath", "seqfma", user_eq=table_oracle.table_rows_at(
        leaves.get("gmath"), event, ALL_ROWS))
    E.set_fd("central")
    xv = problem.xdict_to_vector(x)
    with np.errstate(all="ignore"):
        s, _ = C.sens(helpers.copy_x(x))
    assert_sens_same(s, P.split_jacobian(E.eval_jacobian(xv), key_order=list(x.keys())))


def test_python_refusals():
    Lg = leaves.get("gmath")
    p, u, c, x0 = problem.problem_from_inputs(helpers.example_inputs(), coord=Lg.coordinate_c, max_nodes=12)
    with pytest.raises(ValueError, match="unknown result-table column"):
        gplan.TableAtEvent(AIR_EVENT, [("altitud", 1.0, 0.0)])
    with pytest.raises(ValueError, match="non-zero"):
        gplan.TableAtEvent(AIR_EVENT, [("altitude", 0.0, 0.0)])
    with pytest.raises(ValueError, match="at least one row"):
        gplan.TableAtEvent(AIR_EVENT, [])
    with pytest.raises(KeyError, match="unknown event"):
        gplan.CompiledPlan(p, u, c, user_eq=gplan.TableAtEvent("NO_SUCH_EVENT", [("altitude", 1.0, 0.0)]))
    with pytest.raises(ValueError, match="no first node"):
        gplan.CompiledPlan(p, u, c, user_ineq=gplan.TableAtEvent("SIMEND", [("altitude", 1.0, 0.0)]))
    for bad in (lambda *a: 0.0, [gplan.PerigeeAtEvent("IIP_END"), lambda *a: 0.0], []):
        with pytest.raises(TypeError, match="OrbitAtEvent.*TableAtEvent"):
            gplan.CompiledPlan(p, u, c, user_eq=bad)


def test_c_abi_refuses_out_of_range_job_tables():
    """validate_desc (plan_host.h), which gelato_plan_create runs before anything is uploaded: every index of the job
    tables checked against the plan."""
    p, u, c, x0, O, P = _setup(MIXED_EQ, MIXED_INEQ)
    L = ctypes.CDLL(emu_binding.build())
    L.emu_packed_map.restype = ctypes.c_longlong
    L.emu_packed_map.argtypes = [ctypes.POINTER(engine.PlanDesc), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    assert L.emu_packed_map(ctypes.byref(engine.make_desc(P)[0]), None, None, None) > 0
    cases = [("tab_col", 0, 34), ("tab_col", 1, -1), ("tab_aux", 0, P.n_vals - 17),
             ("tab_aux", 2, -1), ("tab_i32", (0, gplan.GT_TIDX), P.S), ("tab_i32", (1, gplan.GT_SROW), P.M),
             ("tab_i32", (0, gplan.GT_ROW), P.n_rows - 1), ("tab_i32", (1, gplan.GT_NROW), 0),
             ("tab_i32", (1, gplan.GT_R0), P.n_tab_rows), ("tab_i32", (0, gplan.GT_RC0 + 11), -1)]
    for name, at, value in cases:
        orig = getattr(P, name).copy()
        getattr(P, name)[at] = value
        try:
            d, keep = engine.make_desc(P)
            assert L.emu_packed_map(ctypes.byref(d), None, None, None) == -1, (name, at, value)
        finally:
            setattr(P, name, orig)
    d, keep = engine.make_desc(P)
    d.n_tab_rows = P.n_tab_rows - 1
    assert L.emu_packed_map(ctypes.byref(d), None, None, None) == -1
    d.n_tab_rows, d.tab_col = P.n_tab_rows, ctypes.cast(None, ctypes.POINTER(ctypes.c_int32))
    assert L.emu_packed_map(ctypes.byref(d), None, None, None) == -1


def test_one_problem_sharded_the_range_from_block_zero_evaluates_the_table_jobs():
    p, u, c, x0, O, P = _setup(MIXED_EQ, MIXED_INEQ)
    E = emu_table.TableEmulator(P)
    nb, nv = E.block_counts()
    xv = problem.xdict_to_vector(helpers.perturbed(x0))
    g_full, pk_full = E.eval_pair(xv, packed=True)
    g, pk = np.full(P.n_rows, np.nan), np.full(E.n_pack, np.nan)
    E.eval_pair_range(xv, g, pk, (nb // 2, nb), (0, nv))
    tab_slots = np.concatenate([np.arange(E.n_pack - 18 * P.n_tab_rows, E.n_pack)])
    assert np.isnan(pk[tab_slots]).all()
    E.eval_pair_range(xv, g, pk, (0, nb // 2), (0, 0))
    assert _same(g, g_full) and _same(pk, pk_full)


def test_eval_counts():
    p, u, c, x0, O, P = _setup(MIXED_EQ, MIXED_INEQ)
    Lg = leaves.get("gmath")
    Q = gplan.CompiledPlan(p, u, c, user_eq=gplan.PerigeeAtEvent("IIP_END"), coord=Lg.coordinate_c)
    a, b = P.eval_counts(), Q.eval_counts()
    assert a["objfunc"] - b["objfunc"] == 3 and a["sens"] - b["sens"] == 3 * 18


# ---------------------------------------------------------------------------------------------------- GPU tier
def _engine_case(variant="example", factor=1, central=False):
    p, u, c, x0, O, P = _setup(MIXED_EQ, MIXED_INEQ, variant=variant, factor=factor, central=central)
    return p, u, c, x0, O, P


@pytest.mark.gpu
@pytest.mark.parametrize("central", [False, True])
def test_gpu_every_entry_point(central):
    import torch

    p, u, c, x0, O, P = _engine_case(central=central)
    Em = emu_table.TableEmulator(P)
    E = engine.Engine(P)
    if central:
        Em.set_fd("central")
        E.set_fd("central")
    X = np.stack([problem.xdict_to_vector(helpers.perturbed(x0, seed=k)) for k in range(3)])
    g_ref = Em.eval_residuals(X, 3)
    v_ref = Em.eval_jacobian(X, 3)
    _, pk_ref = Em.eval_pair(X, 3, packed=True)
    assert _same(E.eval_residuals(X, 3), g_ref) and _same(E.eval_jacobian(X, 3), v_ref)
    assert _same(E.eval_residuals(X[0]), g_ref[0])  # one scenario: the captured graph
    assert _same(E.eval_residuals(X, 3, scen_ids=[0, 0, 0]), g_ref) and _same(E.eval_jacobian(X, 3, scen_ids=[0, 0, 0]), v_ref)
    g, pk = E.eval_pair_packed(X, 3)
    assert _same(g, g_ref) and _same(pk, pk_ref)
    assert _same(E.eval_jacobian_packed(X, 3), pk_ref)
    for pinned in (False, True):
        if pinned:
            pv, pg, px = engine.PinnedArray(3 * P.n_vals), engine.PinnedArray(3 * P.n_rows), engine.PinnedArray(X.size)
            vals, gg, xx = pv.array, pg.array, px.array
            xx[:] = X.ravel()
        else:
            vals, gg, xx = np.empty(3 * P.n_vals), np.empty(3 * P.n_rows), X.ravel().copy()
        E.jacobian_template(vals, 3)
        E.eval_jacobian_update(xx, vals, 3)
        assert _same(vals.reshape(3, -1), v_ref)
        E.eval_pair_update(xx, gg, vals, 3)
        assert _same(gg.reshape(3, -1), g_ref) and _same(vals.reshape(3, -1), v_ref)
        assert _same(E.eval_residuals(xx, 3, out=gg).reshape(3, -1), g_ref)
    xd = torch.from_numpy(X).cuda()
    gd = torch.full((3, P.n_rows), float("nan"), dtype=torch.float64, device="cuda")
    vd = torch.full((3, P.n_vals), float("nan"), dtype=torch.float64, device="cuda")
    pd = torch.full((3, E.n_pack), float("nan"), dtype=torch.float64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    E.eval_residuals_dev(xd.data_ptr(), gd.data_ptr(), 3, st)
    torch.cuda.synchronize()
    assert _same(gd.cpu().numpy(), g_ref)
    E.fill_template(vd.data_ptr(), 3, st)
    E.eval_jacobian_dev(xd.data_ptr(), vd.data_ptr(), 3, st)
    torch.cuda.synchronize()
    assert _same(vd.cpu().numpy(), v_ref)
    gd.fill_(float("nan"))
    E.eval_pair_dev(xd.data_ptr(), gd.data_ptr(), vd.data_ptr(), 3, st)
    torch.cuda.synchronize()
    assert _same(gd.cpu().numpy(), g_ref) and _same(vd.cpu().numpy(), v_ref)
    gd.fill_(float("nan"))
    E.eval_pair_packed_dev(xd.data_ptr(), gd.data_ptr(), pd.data_ptr(), 3, st)
    torch.cuda.synchronize()
    assert _same(gd.cpu().numpy(), g_ref) and _same(pd.cpu().numpy(), pk_ref)
    # and the oracle itself, through GelatoProblem
    prob = callbacks.GelatoProblem(p, u, c, user_eq=[_builtin(*s) for s in MIXED_EQ],
                                   user_ineq=[_builtin(*s) for s in MIXED_INEQ], coord=leaves.get("gmath").coordinate_c,
                                   derivative="central" if central else "forward")
    x = helpers.perturbed(x0, seed=5)
    with np.errstate(all="ignore"):
        assert_funcs_same(O.objfunc(helpers.copy_x(x))[0], prob.objfunc(x)[0])
        assert_sens_same(O.sens(helpers.copy_x(x))[0], prob.sens(x)[0])
    prob.close()
    E.close()


@pytest.mark.gpu
def test_gpu_plan_without_table_jobs_launches_nothing_new_and_refusals_leave_nothing():
    p, u, c, x0, O, P = _engine_case()
    Lg = leaves.get("gmath")
    Q = gplan.CompiledPlan(p, u, c, user_eq=gplan.PerigeeAtEvent("IIP_END"), coord=Lg.coordinate_c)
    E, F = engine.Engine(P), engine.Engine(Q)
    xv = problem.xdict_to_vector(x0)
    for eng, extra in ((F, 0), (E, 1)):
        n0 = eng.launches
        eng.eval_residuals(np.stack([xv, xv]), 2, scen_ids=[0, 0])  # not the captured graph: one launch per kernel
        eng.eval_jacobian(xv)
        assert eng.launches - n0 == 1 + extra + 2 + extra
    E.close()
    F.close()
    P.tab_col[0] = 34
    with pytest.raises(engine.GelatoError, match="unknown result-table column code"):
        engine.Engine(P)


@pytest.mark.gpu
def test_gpu_dispersed_batch_of_64():
    """Thrust, wind and the mass unit of each scenario enter thrust, dynamic_pressure and accel_BODY_X."""
    Lg = leaves.get("gmath")
    rows = [("thrust", 1e5, 0.0), ("dynamic_pressure", 1e4, 0.0), ("accel_BODY_X", 9.8, 0.0), ("downrange", 1e4, 0.0)]
    plans, xs = [], []
    for k, si in enumerate(scenarios.disperse(helpers.example_inputs(), 64, seed=20260117)):
        p, u, c, x0 = problem.problem_from_inputs(si, coord=Lg.coordinate_c, max_nodes=12)
        plans.append(gplan.CompiledPlan(p, u, c, user_eq=gplan.TableAtEvent("ZEROLIFT_START", rows),
                                        user_ineq=gplan.TableAtEvent(AIR_EVENT, rows[:2]), coord=Lg.coordinate_c))
        xs.append(problem.xdict_to_vector(helpers.perturbed(x0, seed=k)))
        if k < 3:  # a few against the oracle directly
            O = nlp.OracleNLP(p, u, c, "gmath", "seqfma", user_eq=table_oracle.table_rows_at(Lg, "ZEROLIFT_START", rows),
                              user_ineq=table_oracle.table_rows_at(Lg, AIR_EVENT, rows[:2]))
            xd = problem.vector_to_xdict(xs[-1], p["M"], p["N"], p["num_sections"])
            E1 = engine.Engine(plans[-1])
            assert_funcs_same(O.objfunc(helpers.copy_x(xd))[0], plans[-1].split_residuals(E1.eval_residuals(xs[-1])))
            assert_sens_same(O.sens(helpers.copy_x(xd))[0], plans[-1].split_jacobian(E1.eval_jacobian(xs[-1])))
            E1.close()
    X = np.stack(xs)
    E = engine.Engine(plans[0], scenario_plans=plans)
    Em = emu_table.TableEmulator(plans[0], scenario_plans=plans)
    assert _same(E.eval_residuals(X, 64), Em.eval_residuals(X, 64))
    assert _same(E.eval_jacobian(X, 64), Em.eval_jacobian(X, 64))
    g, pk = E.eval_pair_packed(X, 64)
    g2, pk2 = Em.eval_pair(X, 64, packed=True)
    assert _same(g, g2) and _same(pk, pk2)
    # the thrust row differs between scenarios: the per-scenario section parameters reach it
    G = E.eval_residuals(X, 64)
    assert np.unique(G[:, plans[0].group_rows["eqcon_user"][0]]).size > 32
    E.close()


@pytest.mark.gpu
def test_gpu_bench_workload_sample():
    import bench

    plans, X, probs = bench.load_workload("example", 15, 128, 0, 16)  # the first 16 of the step's 128 scenarios
    tplans = [gplan.CompiledPlan(p, u, c, user_eq=[gplan.PerigeeAtEvent("IIP_END"),
                                                   gplan.TableAtEvent("FAIRING", [("altitude", 1e5, 1.0)])],
                                 user_ineq=gplan.TableAtEvent(AIR_EVENT, [("dynamic_pressure", 1e4, 0.0)]))
              for p, u, c, x in probs]
    E = engine.Engine(tplans[0], scenario_plans=tplans)
    G = E.eval_residuals(X, 16)
    g, pk = E.eval_pair_packed(X, 16)
    assert _same(g, G)
    for k in (0, 13):
        Em = emu_table.TableEmulator(tplans[k])
        g1, pk1 = Em.eval_pair(X[k], packed=True)
        assert _same(G[k], g1) and _same(pk[k], pk1)
    E.close()


@pytest.mark.gpu
def test_gpu_residuals_without_the_captured_graph():
    code = ("import sys, numpy as np; sys.path[:0] = [%r, %r]; import test_user_table as t; "
            "print(t._graph_check())") % (os.path.dirname(HERE), HERE)
    env = dict(os.environ, GELATO_B200_NO_GRAPH="1")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and out.stdout.strip().endswith("True"), out.stderr[-2000:]
    assert _graph_check()


def _graph_check():
    p, u, c, x0, O, P = _engine_case()
    E = engine.Engine(P)
    ok = True
    for k in range(3):
        xv = problem.xdict_to_vector(helpers.perturbed(x0, seed=k))
        ok &= _same(E.eval_residuals(xv), emu_table.TableEmulator(P).eval_residuals(xv))
    E.close()
    return bool(ok)


@pytest.mark.gpu
def test_gpu_values_are_the_result_table_columns():
    """(g_r + offset) * scale equals output.kernel_rows on the node's inputs to the rounding of that expression, and a
    row with scale 1 and offset 0 is the column itself, bit for bit."""
    Lg = leaves.get("gmath")
    p, u, c, x0 = problem.problem_from_inputs(helpers.example_inputs(), coord=Lg.coordinate_c, max_nodes=12)
    plain = [(col, 1.0, 0.0) for col in output.KERNEL_COLUMNS]
    for event in (AIR_EVENT, VACUUM_EVENT):
        P = gplan.CompiledPlan(p, u, c, user_eq=gplan.TableAtEvent(event, ALL_ROWS),
                               user_ineq=gplan.TableAtEvent(event, plain), coord=Lg.coordinate_c)
        E = engine.Engine(P)
        x = helpers.perturbed(x0)
        f = P.split_residuals(E.eval_residuals(problem.xdict_to_vector(x)))
        i = p["event_index"][event]
        a = p["ps_params"].index_start_u(i) + i
        prm = p["params"][i]
        inputs = (x["mass"][a: a + 1] * u["mass"], (x["position"][3 * a: 3 * a + 3] * u["position"]).reshape(1, 3),
                  (x["velocity"][3 * a: 3 * a + 3] * u["velocity"]).reshape(1, 3), x["quaternion"][4 * a: 4 * a + 4].reshape(1, 4),
                  x["t"][i: i + 1] * u["t"], np.array([prm["thrust"]]), np.array([prm["reference_area"]]),
                  np.array([prm["nozzle_area"]]))
        ref = output.kernel_rows([np.ascontiguousarray(v, dtype=np.float64) for v in inputs], p["wind_table"], p["ca_table"],
                                 p["LaunchCondition"]["lat"], p["LaunchCondition"]["lon"])[0]
        assert _same(f["ineqcon_user"], ref)
        scale = np.array([r[1] for r in ALL_ROWS])
        offset = np.array([r[2] for r in ALL_ROWS])
        back = (f["eqcon_user"] + offset) * scale
        fin = np.isfinite(ref)
        assert _same(np.isnan(back), np.isnan(ref))
        bound = 4 * np.spacing(np.abs(ref[fin]) + np.abs(offset[fin] * scale[fin]) + 1e-300)
        assert np.all(np.abs(back[fin] - ref[fin]) <= bound)
        E.close()
