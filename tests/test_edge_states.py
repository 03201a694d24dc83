"""Edge-state parity: the kernels against the oracle at decision vectors where rows go non-finite or the per-thread
code sits on a branch edge (DESIGN.md section 8, "edge tier").

Every other parity test feeds trajectories (x0, 1e-3 perturbations, dispersions, the recorded solution), so branch
edges are reached only by chance, and `np.array_equal` cannot compare a NaN slot.  Here each entry of `CATALOGUE`
plants one edge into the variant's x0 -- values only: sizes, ordering and every index the plan compiled stay -- and
the results are compared with `assert_funcs_same` / `assert_sens_same`: equal bits, or NaN on both sides (the payload
is ignored: the device's canonical NaN is not x86's); signed zeros must match.

CPU tier: the host emulator of the kernels (tests/emu) against the oracle (gmath leaves, sequential-FMA D.X):
objfunc / sens, the drop-in callbacks (update mode, fused pair), pair and packed outputs, central differences, the
mesh error estimate and the path check; and the refusal of one-row wind / CA tables by the leaf entry points.
GPU tier: the same catalogue through the CUDA library, and the leaf kernels on edge inputs.
"""
import ctypes

import numpy as np
import pytest

import central_oracle
import emu_binding
import emu_path
import helpers
import mesh_oracle
import path_oracle
from gelato_b200 import callbacks, engine, mesh, problem
from gelato_b200.plan import GS_FLAGS, GSF_AIR, GSF_ENGINE_ON
from oracle import leaves

VARIANTS = ["example", "all_aero", "neg_area", "three_stage", "iip_orbital"]
OMEGA = 7.2921151467e-5  # physics.h: P_OMEGA


# ------------------------------------------------------------------------------------------------ comparator
def _same(a, b):
    """(ok, detail): equal shapes and, element by element, equal bits or NaN on both sides."""
    a = np.ascontiguousarray(np.atleast_1d(np.asarray(a, dtype=np.float64)))
    b = np.ascontiguousarray(np.atleast_1d(np.asarray(b, dtype=np.float64)))
    if a.shape != b.shape:
        return False, ("shape", a.shape, b.shape)
    ok = (a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))
    if ok.all():
        return True, None
    bad = np.flatnonzero(~ok.ravel())
    return False, (int(bad.size), int(bad[0]), float(a.ravel()[bad[0]]), float(b.ravel()[bad[0]]))


def assert_funcs_same(fa, fb):
    """helpers.assert_funcs_equal with the NaN rule above."""
    assert list(fa.keys()) == list(fb.keys())
    for k in fa:
        assert (fa[k] is None) == (fb[k] is None), k
        if fa[k] is not None:
            ok, why = _same(fa[k], fb[k])
            assert ok, (k, why)


def assert_sens_same(sa, sb):
    """helpers.assert_sens_equal with the NaN rule above: same groups, variable order, (row, col) arrays and dtype,
    shapes; values equal bit for bit or NaN on both sides."""
    assert list(sa.keys()) == list(sb.keys())
    for k in sa:
        a, b = sa[k], sb[k]
        assert (a is None) == (b is None), k
        if a is None:
            continue
        assert list(a.keys()) == list(b.keys()), (k, list(a.keys()), list(b.keys()))
        for var in a:
            av, bv = a[var], b[var]
            assert isinstance(av, dict) == isinstance(bv, dict), (k, var)
            if isinstance(av, dict):
                assert tuple(av["shape"]) == tuple(bv["shape"]), (k, var)
                for i in range(2):
                    assert av["coo"][i].dtype == np.int32 and bv["coo"][i].dtype == np.int32, (k, var)
                    assert np.array_equal(av["coo"][i], bv["coo"][i]), (k, var, "index %d" % i)
                ok, why = _same(av["coo"][2], bv["coo"][2])
            else:
                ok, why = _same(av, bv)
            assert ok, (k, var, why)


def test_comparator_rules():
    nan2 = np.array([0x7FF8000000000001], dtype=np.uint64).view(np.float64)[0]  # another NaN payload
    assert _same([np.nan, 1.0], [nan2, 1.0])[0] and _same([-np.nan], [np.nan])[0]
    assert not _same([0.0], [-0.0])[0]
    assert not _same([np.nan], [0.0])[0] and not _same([np.inf], [np.nan])[0]
    assert not _same([1.0, 2.0], [1.0])[0]
    with pytest.raises(AssertionError):
        assert_sens_same({"g": {"m": np.zeros((1, 2))}}, {"g": {"m": np.array([[0.0, np.nan]])}})


# ------------------------------------------------------------------------------------------------ catalogue
def _rows(plan, sec):
    """State rows (node indices into mass / position / ...) of section `sec`."""
    _, _, xa, xb, _ = plan.ps.get_index(sec)
    return list(range(xa, xb))


def _air_rows(plan):
    """State rows of the air sections, those carrying aero rows first."""
    aero = sorted({int(j[1]) for j in plan.aero_i32 if j[2] > 1})
    air = [i for i in range(plan.S) if plan.sec_i32[i, GS_FLAGS] & GSF_AIR and i not in aero]
    return [r for i in aero + air for r in _rows(plan, i)[1:]]


def _air_node(plan):
    """A node inside an air section -- one whose aero rows cover every node ("all") where the variant has such."""
    return _air_rows(plan)[1]


def _coast_vacuum_node(plan):
    """A node of the first section that is both engine-off and out of the air (the vacuum coast); where there is none
    (neg_area: its stage-2 coasts take the air formula) the first engine-off section."""
    off = [i for i in range(plan.S) if not plan.sec_i32[i, GS_FLAGS] & GSF_ENGINE_ON]
    vac = [i for i in off if not plan.sec_i32[i, GS_FLAGS] & GSF_AIR]
    return _rows(plan, (vac or off)[0])[1]


def _geopotential_altitude(pos_m):
    """physics.h: pos_part -- the geopotential altitude of the geodetic altitude of the ECI position (quirk A.5-2)."""
    L = leaves.get("gmath")
    return L.USStandardAtmosphere_c.geopotential_altitude(L.coordinate_c.ecef2geodetic(*pos_m)[2])


_PLACED = {}


def _put_altitude(x, plan, row, h):
    """Move node `row`'s position until its geopotential altitude reaches h: bisection over a radial scale (the first
    scale found whose altitude is >= h), then a search over single-ulp steps of the two largest components for h
    itself.  The geodetic altitude is a difference of two ~6.4e6 m values, on a grid of 2^-30 m, so h is hit exactly
    where the grid holds it (the bases of 86 km and up, where geopotential = geometric altitude); below 86 km the
    geopotential conversion moves off that grid and the node sits within 1e-8 m above the base.  Memoised."""
    p = x["position"][3 * row: 3 * row + 3].copy()
    key = (p.tobytes(), h, plan.units[1])
    if key not in _PLACED:
        alt = lambda q: _geopotential_altitude(q * plan.units[1])  # noqa: E731
        lo, hi = 0.5, 2.0
        for _ in range(200):
            mid = 0.5 * (lo + hi)
            if mid in (lo, hi):
                break
            lo, hi = (mid, hi) if alt(p * mid) < h else (lo, mid)
        base = p * hi
        a, b = np.argsort(-np.abs(base))[:2]
        _PLACED[key] = base
        for i, j in sorted(((i, j) for i in range(-8, 9) for j in range(-8, 9)), key=lambda ij: abs(ij[0]) + abs(ij[1])):
            q = base.copy()
            q[a] += i * np.spacing(q[a])
            q[b] += j * np.spacing(q[b])
            if alt(q) == h:
                _PLACED[key] = q
                break
    x["position"][3 * row: 3 * row + 3] = _PLACED[key]


def _earth_fixed_velocity(x, plan, row):
    """ECI velocity of node `row` = omega x r: zero velocity relative to the rotating Earth."""
    r = x["position"][3 * row: 3 * row + 3] * plan.units[1]
    x["velocity"][3 * row: 3 * row + 3] = np.array([-OMEGA * r[1], OMEGA * r[0], 0.0]) / plan.units[2]


def _edge(fn):
    def make(x0, plan):
        x = helpers.copy_x(x0)
        fn(x, plan)
        return x
    make.__doc__ = fn.__doc__
    return make


US76_BASES = (11000.0, 20000.0, 32000.0, 47000.0, 51000.0, 71000.0, 86000.0, 91000.0, 110000.0, 120000.0)
SPECIALS = np.array([0.9999999999, 0.249999995, 3e-9, 1e-12, 0.0, 0.499999999, -3e-9, 1.0 - 1e-9])


def _set(key, sl, value):
    def f(x, plan):
        x[key][sl] = value
    return f


def _node(key, width, value, where=None):
    def f(x, plan):
        r = (where or _air_node)(plan)
        x[key][width * r: width * r + width] = value
    return f


def _scale_node(key, width, factor):
    def f(x, plan):
        r = _air_node(plan)
        x[key][width * r: width * r + width] *= factor
    return f


def _us76_bases(x, plan):
    """Geopotential altitude on each US-76 layer base (physics.h: us76_layer, us76), one air node each."""
    for row, h in zip(_air_rows(plan), US76_BASES):
        _put_altitude(x, plan, row, h)


def _wind_knots(x, plan):
    """Altitude on each interior knot of the wind table (physics.h: interp_interval, pos_part's interpolation), one air
    node each."""
    knots = plan.wind[1:-1, 0]
    for row, h in zip(_air_rows(plan)[len(US76_BASES):], knots):
        _put_altitude(x, plan, row, h)


def _mach_zero(x, plan):
    """Zero air-relative velocity below 1 km (no wind there): Mach 0, the CA table's first knot (physics.h:
    rhs_velocity_air_col, interp_table), and the aero rows' angle of attack of a zero vector (aero_quantity_col)."""
    _earth_fixed_velocity(x, plan, 1)


def _residue_and_nonfinite(x, plan):
    """Residue-sensitive values ((x + dx) - dx != x, DESIGN.md H3) in velocity / quaternion / u, with a NaN mass and
    an infinite control at other nodes (jobs.h: residue, residue_n; the NaN rows of the dynamics)."""
    rng = np.random.default_rng(3)
    for k in ("velocity", "quaternion", "u"):
        idx = rng.choice(x[k].size, size=24, replace=False)
        x[k][idx] = rng.choice(SPECIALS, size=24)
    x["mass"][7] = np.nan
    x["u"][9] = np.inf


# name -> (make(x0, plan) -> xdict, NaN-producing: a NaN in the shipped example's objfunc rows or sens values); each
# comment names the code path the entry reaches
CATALOGUE = {
    # jobs.h: time_node / the t columns of every block: a section of zero and of negative length
    "dt_zero": (_edge(lambda x, p: x["t"].__setitem__(3, x["t"][2])), False),
    "dt_negative": (_edge(lambda x, p: x["t"].__setitem__(3, x["t"][2] - 1e-3)), False),
    # jobs.h: time_node -> Earth-rotation angle inf (gmath.h: gm_sincos of inf)
    "t_final_inf": (_edge(_set("t", -1, np.inf)), True),
    # physics.h: rhs_velocity_air_col thrust / mass, H5 shared reciprocal of a zero and a signed-zero divisor
    "mass_zero": (_edge(_node("mass", 1, 0.0)), True),
    "mass_negative_zero": (_edge(_node("mass", 1, -0.0)), False),
    "mass_negative": (_edge(_node("mass", 1, -0.3)), False),
    # physics.h: rhs_velocity_noair_col on a coast (thrust 0): noair_div_by's zero numerator over a negative mass
    "coast_mass_negative": (_edge(_node("mass", 1, -0.5, _coast_vacuum_node)), False),
    "coast_mass_negative_zero": (_edge(_node("mass", 1, -0.0, _coast_vacuum_node)), True),
    # every row that reads the mass: NaN propagation
    "mass_nan": (_edge(_set("mass", 7, np.nan)), True),
    # gmath.h: gm_div_by / gm_rcp outside the +-500 exponent window (H5 guard: plain division)
    "mass_tiny": (_edge(lambda x, p: x["mass"].__imul__(1e-160)), True),
    "position_tiny": (_edge(_scale_node("position", 3, 1e-200)), False),
    # physics.h: quatrot / rhs_quaternion / aero_quantity_col with a zero and a negated attitude quaternion
    "quaternion_zero_node": (_edge(_node("quaternion", 4, 0.0)), True),
    "quaternion_zero_all": (_edge(_set("quaternion", slice(None), 0.0)), True),
    "quaternion_negated": (_edge(lambda x, p: x["quaternion"].__imul__(-1.0)), False),
    # physics.h: air_velocity, aero_quantity_col (acos / atan2 of a zero vector); orbit_quantity (user rows)
    "velocity_zero_node": (_edge(_node("velocity", 3, 0.0)), False),
    "velocity_zero_all": (_edge(_set("velocity", slice(None), 0.0)), True),  # the user row is NaN (jac_fd's blocks)
    "velocity_nan_node": (_edge(_node("velocity", 3, np.nan)), True),
    # physics.h: Mach far past the CA table's last knot (interp_interval -> -2)
    "velocity_x50": (_edge(_scale_node("velocity", 3, 50.0)), False),
    # physics.h: air_velocity == 0 at a node carrying aero rows (ECI velocity = omega x r)
    "air_relative_zero": (_edge(lambda x, p: _earth_fixed_velocity(x, p, _air_node(p))), False),
    "mach_zero_on_first_ca_knot": (_edge(_mach_zero), False),
    # physics.h: rhs_quaternion with an infinite rate
    "u_inf": (_edge(_set("u", 4, np.inf)), False),
    # physics.h: ecef2geodetic at the pole (x = y = 0) and at the Earth's centre; gravity_eci of r = 0
    "position_pole": (_edge(_node("position", 3, [0.0, 0.0, 1.0])), False),
    "position_origin": (_edge(_node("position", 3, 0.0)), False),
    # physics.h: us76 above 86 km (geometric = geopotential), below 0 m and far out
    "altitude_above_86km": (_edge(_scale_node("position", 3, 1.02)), False),
    "altitude_negative": (_edge(_scale_node("position", 3, 0.99)), False),
    "altitude_all_x1.5": (_edge(lambda x, p: x["position"].__imul__(1.5)), False),
    # physics.h: interp_interval above the wind table's last knot (1e10 m)
    "altitude_past_wind_table": (_edge(_scale_node("position", 3, 2000.0)), False),
    "altitude_on_us76_bases": (_edge(_us76_bases), False),
    "altitude_on_wind_knots": (_edge(_wind_knots), False),
    # jobs.h: residue / residue_n with non-finite neighbours
    "residue_and_nonfinite": (_edge(_residue_and_nonfinite), True),
}
CASES = list(CATALOGUE)
# the subset central differences and the GPU's central mode run (each of these reaches a different branch)
CENTRAL_CASES = ["dt_zero", "coast_mass_negative", "mass_nan", "velocity_zero_all", "air_relative_zero",
                 "position_origin", "altitude_on_us76_bases", "residue_and_nonfinite"]

_CACHE = {}


def _setup(variant):
    """(p, u, c, x0, oracle, plan) of a variant at max_nodes = 12 (built once per session)."""
    if variant not in _CACHE:
        Lg = leaves.get("gmath")
        p, u, c, x0 = problem.problem_from_inputs(helpers.variant_inputs(variant), coord=Lg.coordinate_c, max_nodes=12)
        _CACHE[variant] = (p, u, c, x0, helpers.oracle_nlp(p, u, c, "gmath", "seqfma"),
                           helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c))
    return _CACHE[variant]


def _oracle(O, x):
    """(funcs, funcsSens) of the oracle at x (its sens perturbs its own copy in place)."""
    with np.errstate(all="ignore"):
        xa = helpers.copy_x(x)
        f, _ = O.objfunc(xa)
        s, _ = O.sens(xa)
    return f, s


def test_catalogue_reaches_its_edges():
    """The planted values are where the names say, every entry keeps the sizes, and the NaN-producing flags hold."""
    p, u, c, x0, O, P = _setup("example")
    for name, (make, nan) in CATALOGUE.items():
        x = make(x0, P)
        assert list(x) == list(x0) and all(x[k].shape == x0[k].shape for k in x), name
        assert any(not np.array_equal(x[k], x0[k]) for k in x), name
        f, s = _oracle(O, x)
        vals = [np.asarray(v, dtype=np.float64) for v in f.values() if v is not None]
        vals += [np.asarray(b["coo"][2] if isinstance(b, dict) else b) for g in s.values() if g for b in g.values()]
        assert any(np.isnan(v).any() for v in vals) == nan, name
    p, u, c, x0, O, P = _setup("all_aero")
    x = CATALOGUE["altitude_on_us76_bases"][0](x0, P)
    rows = _air_rows(P)
    for row, h in zip(rows, US76_BASES):
        got = _geopotential_altitude(x["position"][3 * row: 3 * row + 3] * P.units[1])
        assert h <= got < h + 1e-8 and (got == h or h < 86000.0), (h, got)
    x = CATALOGUE["altitude_on_wind_knots"][0](x0, P)
    for row, h in zip(rows[len(US76_BASES):], P.wind[1:-1, 0]):
        got = _geopotential_altitude(x["position"][3 * row: 3 * row + 3] * P.units[1])
        assert h <= got < h + 1e-8 and (got == h or h < 86000.0), (h, got)
    assert len(rows) >= len(US76_BASES) + P.wind.shape[0] - 2


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("variant", VARIANTS)
def test_emulator_matches_oracle_on_edge_states(variant, case):
    """objfunc rows and every sens value (dense user blocks included) of the kernels' code against the oracle."""
    p, u, c, x0, O, P = _setup(variant)
    E = emu_binding.Emulator(P)
    x = CATALOGUE[case][0](x0, P)
    f, s = _oracle(O, x)
    xv = problem.xdict_to_vector(x)
    assert_funcs_same(f, P.split_residuals(E.eval_residuals(xv)))
    assert_sens_same(s, P.split_jacobian(E.eval_jacobian(xv), key_order=list(x.keys())))


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("variant", VARIANTS)
def test_pair_and_packed_outputs_on_edge_states(variant, case):
    """eval_pair (COO and packed, mapped through packed_map) against the separate residual / Jacobian calls."""
    p, u, c, x0, O, P = _setup(variant)
    E = emu_binding.Emulator(P)
    full, src, sgn = E.packed_map()
    xv = problem.xdict_to_vector(CATALOGUE[case][0](x0, P))
    g_ref, v_ref = E.eval_residuals(xv), E.eval_jacobian(xv)
    g, v = E.eval_pair(xv)
    assert _same(g, g_ref)[0] and _same(v, v_ref)[0]
    g, pk = E.eval_pair(xv, packed=True)
    v = P.vals_template.copy()
    v[full] = sgn * pk[src]
    assert _same(g, g_ref)[0]
    ok, why = _same(v, v_ref)
    assert ok, why


@pytest.mark.parametrize("case", CASES)
def test_drop_in_callbacks_on_edge_states(case):
    """GelatoProblem on the emulator -- update mode (refresh_user_blocks), fresh arrays and the fused pair -- returns
    the oracle's dictionaries, NaN slots of the dense user blocks included."""
    p, u, c, x0, O, P = _setup("example")
    Lg = leaves.get("gmath")
    x = CATALOGUE[case][0](x0, P)
    f, s = _oracle(O, x)
    mk = lambda **kw: callbacks.GelatoProblem(p, u, c, user_eq=callbacks.PerigeeAtEvent(helpers.USER_EVENT),  # noqa: E731
                                              coord=Lg.coordinate_c, engine_factory=emu_binding.EmuEngine, **kw)
    for prob in (mk(), mk(reuse_output=False), mk(fuse_pair=True)):
        prob.sens(x0)  # a finite point first: the kept dictionary is refreshed in place at x
        fg, _ = prob.objfunc(x)
        assert_funcs_same(f, fg)
        assert_sens_same(s, prob.sens(x, fg)[0])


def test_user_blocks_carry_jac_fd_nan_and_csr_keeps_structural_zeros():
    """velocity_zero_all makes the user row NaN: jac_fd's (g_base - g_base)/dx is NaN in every entry of the dense
    blocks, including the variables visited before the first one the function reads.  csr_map keeps those entries as
    structural zeros (DESIGN.md H4): a CSR consumer sees 0 there and NaN in the row's other entries."""
    p, u, c, x0, O, P = _setup("example")
    E = emu_binding.Emulator(P)
    x = CATALOGUE["velocity_zero_all"][0](x0, P)
    vals = E.eval_jacobian(problem.xdict_to_vector(x))
    blk = P.split_jacobian(vals, key_order=list(x.keys()))["eqcon_user"]
    assert all(np.isnan(b).all() for b in blk.values())
    fin = P.split_jacobian(E.eval_jacobian(problem.xdict_to_vector(x0)), key_order=list(x0.keys()))["eqcon_user"]
    assert not np.signbit(fin["mass"]).any() and (fin["mass"] == 0.0).all()  # +0 where g_base is finite
    m = P.csr_map(key_order=list(x.keys()))
    r0 = m["row0"]["eqcon_user"]
    lo, hi = m["indptr"][r0], m["indptr"][r0 + 1]
    data = np.append(vals, 0.0)[m["src"][lo:hi]]
    structural = m["src"][lo:hi] == P.n_vals
    assert structural.sum() == P.sizes["mass"] + 3 * _user_row(P)
    assert (data[structural] == 0.0).all() and np.isnan(data[~structural]).all()


def _user_row(P):
    """The state row the user constraint reads (the first node of its event's section)."""
    return P.blocks["eqcon_user"][2]


@pytest.mark.parametrize("case", CENTRAL_CASES)
@pytest.mark.parametrize("variant", ["example", "all_aero", "three_stage"])
def test_central_mode_matches_central_oracle_on_edge_states(variant, case):
    p, u, c, x0, O, P = _setup(variant)
    from oracle import user_builtin

    Lg = leaves.get("gmath")
    C = central_oracle.CentralOracleNLP(p, u, c, "gmath", "seqfma", user_eq=user_builtin.perigee_ratio_at(Lg, helpers.USER_EVENT))
    E = emu_binding.Emulator(P)
    E.set_fd("central")
    x = CATALOGUE[case][0](x0, P)
    with np.errstate(all="ignore"):
        s, _ = C.sens(helpers.copy_x(x))
    xv = problem.xdict_to_vector(x)
    assert_sens_same(s, P.split_jacobian(E.eval_jacobian(xv), key_order=list(x.keys())))
    full, src, sgn = E.packed_map()
    _, pk = E.eval_pair(xv, packed=True)
    v = P.vals_template.copy()
    v[full] = sgn * pk[src]
    assert _same(v, E.eval_jacobian(xv))[0]


def _mesh_path_want(O, x, tabs):
    with np.errstate(all="ignore"):
        return mesh_oracle.mesh_error(O, x, tabs), path_oracle.path_check(O, x, tabs)


def _assert_nan_rule(res, at):
    """DESIGN.md section 11: a NaN propagates as numpy's min does; `at` is then a test point's index (the first NaN's,
    which the comparison with path_oracle pins)."""
    for j in np.flatnonzero(np.isnan(res)):
        assert at[j] >= 0, j


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("variant", ["example", "all_aero", "three_stage"])
def test_mesh_error_and_path_check_on_edge_states(variant, case):
    """The mesh error estimate and the path check of the kernels' code against tests/mesh_oracle.py and
    tests/path_oracle.py, NaN propagation and the first NaN's index included."""
    p, u, c, x0, O, P = _setup(variant)
    E = emu_path.PathEmuEngine(P)
    tabs = mesh.grid_tables(P.ps)
    E.set_mesh_grid(tabs)
    x = CATALOGUE[case][0](x0, P)
    xv = problem.xdict_to_vector(x)
    err_want, (res_want, at_want) = _mesh_path_want(O, x, tabs)
    err = E.mesh_error(xv)
    ok, why = _same(err, err_want)
    assert ok, why
    res, at = E.path_check(xv)
    ok, why = _same(res, res_want)
    assert ok and np.array_equal(at, at_want), (why, at, at_want)
    _assert_nan_rule(res, at)


# ---- leaf tables: one row is refused before anything touches the device
_pd = ctypes.POINTER(ctypes.c_double)


def test_leaf_entry_points_refuse_one_row_tables():
    """interp_interval / np_interp read rows k and k + 1: every leaf entry point that takes a wind or CA table refuses
    fewer than two rows with GELATO_ERR_ARG and a message, as gelato_plan_create does."""
    L = engine.load_library()
    n = 2
    st = np.zeros((n, 3))
    q = np.tile([1.0, 0.0, 0.0, 0.0], (n, 1))
    one = np.zeros(n)
    prm, un = np.array([420000.0, 140.9, 2.21, 0.0, 0.68]), np.array([27442.0, 6378137.0, 1000.0])
    w1, w2, c1, c2 = np.zeros((1, 3)), np.zeros((2, 3)), np.zeros((1, 2)), np.zeros((2, 2))
    out = np.zeros((n, 64))
    keep = []

    def P(a):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=np.float64)
        keep.append(a)
        return a.ctypes.data_as(_pd)

    def dyn(w, nw, ca, nc):
        return L.gelato_leaf_dynamics_velocity(0, n, P(one), P(st), P(st), P(q), P(one), P(prm), P(w), nw, P(ca), nc, P(un),
                                               P(out))

    def aero(w, nw, kind=1):
        return L.gelato_leaf_aero(0, kind, n, P(st), P(st), P(q), P(one), P(w), nw, P(out))

    def table(w, nw, ca, nc):
        return L.gelato_leaf_output_table(0, n, *[P(a) for a in (one, st, st, q, one, one, one, one)], P(w), nw, P(ca), nc,
                                          0.0, 0.0, P(out))

    def init(w, nw, ca, nc):
        x0, ev, zlt = np.zeros(11), np.zeros((2, 6)), np.zeros(2, dtype=np.int32)
        strides, tout = np.zeros(4, dtype=np.int64), np.array([0.0, 1.0])
        return L.gelato_init_rocket_simulation(0, 1, P(x0), P(ev), zlt.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), 2,
                                               P(np.zeros((3, 4))), 3, P(w), nw, P(ca), nc,
                                               strides.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), 0.0, P(tout), 2, 0.1,
                                               P(np.zeros((1, 2, 11))), None)

    calls = [(lambda: dyn(w1, 1, c2, 2), "wind"), (lambda: dyn(w2, 2, c1, 1), "ca"), (lambda: dyn(None, 2, c2, 2), "wind"),
             (lambda: aero(w1, 1), "wind"), (lambda: aero(w1, 1, kind=4), "wind"), (lambda: aero(w2, 0), "wind"),
             (lambda: table(w1, 1, c2, 2), "wind"), (lambda: table(w2, 2, c1, 1), "ca"),
             (lambda: init(w1, 1, c2, 2), "wind"), (lambda: init(w2, 2, c1, 1), "ca")]
    for call, which in calls:
        assert call() == -1  # GELATO_ERR_ARG
        msg = L.gelato_last_error().decode()
        assert "%s table needs at least two rows" % which in msg, msg


def test_leaf_wrappers_surface_the_one_row_refusal():
    from gelato_b200.lib import dynamics_c, utils_c

    pos, vel, q = np.array([[6.4e6, 0.0, 0.0]]), np.array([[0.0, 400.0, 0.0]]), np.array([[1.0, 0.0, 0.0, 0.0]])
    with pytest.raises(engine.GelatoError, match="wind table needs at least two rows"):
        utils_c.wind_ned(1000.0, [[0.0, 1.0, 2.0]])
    with pytest.raises(engine.GelatoError, match="wind table needs at least two rows"):
        utils_c.dynamic_pressure_array_pa(pos, vel, [0.0], [0.0, 1.0, 2.0])  # a flat row is one row, not three
    with pytest.raises(engine.GelatoError, match="ca table needs at least two rows"):
        dynamics_c.dynamics_velocity([1.0], pos / 6378137.0, vel / 1000.0, q, [0.0], [420000.0, 140.9, 2.21, 0.0, 0.68],
                                     [[0.0, 0.0, 0.0], [1e4, 0.0, 0.0]], [[0.0, 0.3]], [27442.0, 6378137.0, 1000.0])


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.fixture(scope="module")
def gpu_problems():
    made = {}

    def get(variant, derivative="forward"):
        key = (variant, derivative)
        if key not in made:
            p, u, c, x0, O, P = _setup(variant)
            made[key] = callbacks.GelatoProblem(p, u, c, user_eq=callbacks.PerigeeAtEvent(helpers.USER_EVENT),
                                                coord=leaves.get("gmath").coordinate_c, derivative=derivative)
        return made[key]

    yield get
    for prob in made.values():
        prob.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_gpu_callbacks_match_oracle_on_edge_states(gpu_problems, variant):
    """GelatoProblem.objfunc / sens on the device against the oracle, every catalogue entry."""
    p, u, c, x0, O, P = _setup(variant)
    prob = gpu_problems(variant)
    for case in CASES:
        x = CATALOGUE[case][0](x0, P)
        f, s = _oracle(O, x)
        fg, fail = prob.objfunc(x)
        assert fail is False
        try:
            assert_funcs_same(f, fg)
            assert_sens_same(s, prob.sens(x, fg)[0])
        except AssertionError as e:
            raise AssertionError((case, e.args))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["example", "all_aero", "three_stage"])
def test_gpu_pair_entry_points_on_edge_states(gpu_problems, variant):
    """The whole catalogue as one batch: Engine.eval_pair_packed and gelato_eval_pair_packed_dev / _pair_dev against
    the separate residual and Jacobian calls."""
    import torch

    p, u, c, x0, O, P = _setup(variant)
    E = gpu_problems(variant).engine
    X = np.stack([problem.xdict_to_vector(CATALOGUE[k][0](x0, P)) for k in CASES])
    n = X.shape[0]
    g_want = E.eval_residuals(X, n).reshape(n, -1).copy()
    v_want = E.eval_jacobian(X, n).reshape(n, -1).copy()
    full, src, sgn = E.packed_map()

    def expand(pk):
        v = np.tile(P.vals_template, (n, 1))
        v[:, full] = sgn * pk.reshape(n, -1)[:, src]
        return v

    G, PK = E.eval_pair_packed(X, n)
    for k in range(n):
        assert _same(G.reshape(n, -1)[k], g_want[k])[0], CASES[k]
        assert _same(expand(PK)[k], v_want[k])[0], CASES[k]
    xd = torch.from_numpy(X).cuda()
    gd = torch.full((n, P.n_rows), 0.5, dtype=torch.float64, device="cuda")
    pd = torch.full((n, E.n_pack), 0.5, dtype=torch.float64, device="cuda")
    vd = torch.from_numpy(np.tile(P.vals_template, (n, 1))).cuda()
    gd2 = torch.full((n, P.n_rows), 0.5, dtype=torch.float64, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        E.eval_pair_packed_dev(xd.data_ptr(), gd.data_ptr(), pd.data_ptr(), n, s.cuda_stream)
        E.eval_pair_dev(xd.data_ptr(), gd2.data_ptr(), vd.data_ptr(), n, s.cuda_stream)
    s.synchronize()
    for k in range(n):
        for got, want in ((gd.cpu().numpy()[k], g_want[k]), (expand(pd.cpu().numpy())[k], v_want[k]),
                          (gd2.cpu().numpy()[k], g_want[k]), (vd.cpu().numpy()[k], v_want[k])):
            ok, why = _same(got, want)
            assert ok, (CASES[k], why)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["example", "all_aero", "three_stage"])
def test_gpu_central_mode_on_edge_states(gpu_problems, variant):
    from oracle import user_builtin

    p, u, c, x0, O, P = _setup(variant)
    C = central_oracle.CentralOracleNLP(p, u, c, "gmath", "seqfma",
                                        user_eq=user_builtin.perigee_ratio_at(leaves.get("gmath"), helpers.USER_EVENT))
    prob = gpu_problems(variant, "central")
    for case in CENTRAL_CASES:
        x = CATALOGUE[case][0](x0, P)
        with np.errstate(all="ignore"):
            s, _ = C.sens(helpers.copy_x(x))
        try:
            assert_sens_same(s, prob.sens(x)[0])
        except AssertionError as e:
            raise AssertionError((case, e.args))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["example", "all_aero", "three_stage"])
def test_gpu_mesh_error_and_path_check_on_edge_states(gpu_problems, variant):
    p, u, c, x0, O, P = _setup(variant)
    E = gpu_problems(variant).engine
    tabs = mesh.grid_tables(P.ps)
    E.set_mesh_grid(tabs)
    xs = [CATALOGUE[k][0](x0, P) for k in CASES]
    X = np.stack([problem.xdict_to_vector(x) for x in xs])
    n = X.shape[0]
    err = np.asarray(E.mesh_error(X, n_scen=n)).reshape(n, P.S, 11)
    res, at = E.path_check(X, n_scen=n)
    res, at = np.asarray(res).reshape(n, -1), np.asarray(at).reshape(n, -1)
    for k, x in enumerate(xs):
        err_want, (res_want, at_want) = _mesh_path_want(O, x, tabs)
        assert _same(err[k], err_want)[0], CASES[k]
        assert _same(res[k], res_want)[0] and np.array_equal(at[k], at_want), CASES[k]
        _assert_nan_rule(res[k], at[k])


@pytest.mark.gpu
def test_gpu_leaf_kernels_on_edge_inputs():
    """gelato_leaf_* against leaves.get("gmath") at zero air-relative velocity, the poles, the Earth's centre, and
    altitudes / Mach numbers on table knots and past both ends."""
    from gelato_b200.lib import IIP_c, coordinate_c, dynamics_c, utils_c

    L = leaves.get("gmath")
    inp = helpers.example_inputs()
    wind, ca = np.asarray(inp["wind_table"], dtype=float), np.asarray(inp["ca_table"], dtype=float)
    R = 6378137.0
    pos = np.array([[R + 500.0, 0.0, 0.0], [0.0, 0.0, 6356752.3142], [0.0, 0.0, -6356752.3142 - 3e4], [0.0, 0.0, 0.0],
                    [R * 0.6, R * 0.8, 0.0], [0.0, R + 3e4, 0.0], [R + 2e5, 0.0, 0.0], [R * 1e-9, 0.0, 0.0]])
    t = np.array([0.0, 10.0, 100.0, 0.0, 50.0, 0.0, 300.0, 0.0])
    c_, s_ = np.cos(OMEGA * t), np.sin(OMEGA * t)
    vel = np.stack([-OMEGA * pos[:, 1], OMEGA * pos[:, 0], np.zeros(len(t))], axis=1)  # earth-fixed: zero air speed below 1 km
    vel[5:] += np.array([[0.0, 0.0, 900.0], [7000.0, 0.0, 0.0], [0.0, 1e5, 0.0]])  # Mach 2.9, 23, 300 (past the last knot)
    q = np.tile([1.0, 0.0, 0.0, 0.0], (len(t), 1))
    q[2] = [0.0, 0.0, 0.0, 0.0]

    def eq(a, b, what):
        ok, why = _same(a, b)
        assert ok, (what, why)

    eq(utils_c.angle_of_attack_all_array_rad(pos, vel, q, t, wind), L.utils_c.angle_of_attack_all_array_rad(pos, vel, q, t, wind), "alpha")
    eq(utils_c.dynamic_pressure_array_pa(pos, vel, t, wind), L.utils_c.dynamic_pressure_array_pa(pos, vel, t, wind), "q")
    eq(utils_c.q_alpha_array_pa_rad(pos, vel, q, t, wind), L.utils_c.q_alpha_array_pa_rad(pos, vel, q, t, wind), "qalpha")
    eq(utils_c.angle_of_attack_ab_array_rad(pos, vel, q, t, wind),
       [L.utils_c.angle_of_attack_ab_rad(pos[i], vel[i], q[i], t[i], wind) for i in range(len(t))], "alpha ab")
    alts = np.concatenate([wind[:, 0], [-2e8, 2e10, np.nextafter(0.0, -1.0), np.nextafter(1000.0, 2e3), np.nan]])
    eq(utils_c.wind_ned(alts, wind), [L.utils_c.wind_ned(a, wind) for a in alts], "wind_ned")
    eq(coordinate_c.eci2geodetic(pos, t), [L.coordinate_c.eci2geodetic(p, tt) for p, tt in zip(pos, t)], "eci2geodetic")
    eq(coordinate_c.gravity(pos), [L.coordinate_c.gravity(p) for p in pos], "gravity")
    pe = np.array([L.coordinate_c.eci2ecef(p, tt) for p, tt in zip(pos, t)])
    ve = np.array([L.coordinate_c.vel_eci2ecef(v, p, tt) for v, p, tt in zip(vel, pos, t)])
    ve[1] = 0.0
    for fill in (True, False):
        eq(IIP_c.posLLH_IIP_FAA(pe, ve, fill), np.array([L.IIP_c.posLLH_IIP_FAA(a, b, fill) for a, b in zip(pe, ve)]), "iip")
    units = np.array([27442.0, R, 1000.0])
    mass = np.array([0.5, 0.0, -0.0, -0.3, 0.5, 0.5, 1e-160, 0.5])
    param = np.array([420000.0, 140.9, 2.21, 0.0, 0.68])
    for table in (ca, ca + [[0.5, 0.0]]):  # the shifted table starts above Mach 0: the slow nodes fall below its first knot
        a = (mass, pos / R, vel / 1000.0, q, t / 630.0, param, wind, table, units)
        eq(dynamics_c.dynamics_velocity(*a), L.dynamics_c.dynamics_velocity(*a), "dynamics_velocity")
    b = (mass, pos / R, q, np.array([0.0, 140.9, 2.21, 0.0, 0.68]), units)  # thrust 0: a coast, zero numerators
    eq(dynamics_c.dynamics_velocity_NoAir(*b), L.dynamics_c.dynamics_velocity_NoAir(*b), "dynamics_velocity_NoAir")
