"""Sections made of several LGR intervals: h-refinement with per-interval error estimates (DESIGN.md section 11).

CPU tier: the composite differentiation matrix, the NLP kernels' code in the host emulator on composite meshes against
the oracle bit for bit (forward and central) with the layout of the same node counts, the per-interval estimate
against tests/mesh_intervals_oracle.py bit for bit, its square-grid identity and h-convergence, grid refusals, refine_nodes'
ph rule, transfer, the path check and path rows on composite grids, and the host users of tau.  GPU tier: the same
parity through the C ABI (pair, packed and update modes too), the per-interval estimate on a dispersed batch, through
host / pinned / device buffers, and a benchmark-workload sample with two sections split."""
import copy
import ctypes

import numpy as np
import pytest

import emu_binding
import emu_intervals
import helpers
import mesh_intervals_oracle
import mesh_oracle
import path_oracle
import path_rows_oracle
from central_oracle import CentralOracleNLP
from gelato_b200 import engine, initialize, mesh, nlpshim, output, problem, scenarios
from gelato_b200.psparams import PSparams, lgr_diff_matrix, lgr_nodes, mesh_tables
from oracle import leaves, user_builtin
from test_mesh_error import _coast_state

EPS = np.finfo(np.float64).eps

# event name -> (interval counts, breaks or None)
SPLITS = {
    "zl_8_8": {"ZEROLIFT_START": ([8, 8], None)},
    "zl_3_unequal": {"ZEROLIFT_START": ([5, 6, 5], [-0.6, 0.2])},
    "coast": {"SECO": ([3, 3], None), "SEP2": ([2, 1], [0.3])},
}


def _bits(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64)).view(np.int64)


def _eq(a, b):
    return np.shape(a) == np.shape(b) and np.array_equal(_bits(a), _bits(b))


def _with_intervals(inp, splits, factor=1):
    """inputs whose events in `splits` are made of LGR intervals (factor > 1: the benchmark's refined mesh first)."""
    inp = copy.deepcopy(inp)
    if factor != 1:
        inp["events"], inp["settings"]["FlightConstraint"] = problem.refine_events(
            inp["events"], inp["settings"]["FlightConstraint"], factor, 20)
    for e in inp["events"]:
        if e["name"] in splits:
            counts, breaks = splits[e["name"]]
            e["num_nodes"] = sum(counts)
            e["mesh_intervals"] = list(counts)
            if breaks is not None:
                e["mesh_breaks"] = list(breaks)
    return inp


def _plain(inp):
    """the same node counts without intervals"""
    inp = copy.deepcopy(inp)
    for e in inp["events"]:
        e.pop("mesh_intervals", None)
        e.pop("mesh_breaks", None)
    return inp


_CACHE = {}


def _setup(name, derivative="forward"):
    key = (name, derivative)
    if key not in _CACHE:
        Lg = leaves.get("gmath")
        inp = _with_intervals(helpers.example_inputs(), SPLITS[name])
        p, u, c, x0 = problem.problem_from_inputs(inp, coord=Lg.coordinate_c)
        ue = user_builtin.perigee_ratio_at(Lg, helpers.USER_EVENT)
        O = CentralOracleNLP(p, u, c, "gmath", "seqfma", user_eq=ue, derivative=derivative)
        _CACHE[key] = (inp, p, u, c, x0, O, helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c))
    return _CACHE[key]


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("counts,breaks", [([8, 8], None), ([2, 1, 3], [-0.5, 0.25]), ([1, 4], [-0.9]), ([3, 3, 3, 3], None)])
def test_composite_differentiation_matrix(counts, breaks):
    n = sum(counts)
    ps = PSparams([n], [(counts, breaks)])
    D, tau = ps.D(0), ps.tau(0)
    got_counts, b_in, cols = ps.intervals(0)
    assert got_counts == counts and cols == list(np.concatenate(([0], np.cumsum(counts)[:-1])))
    b = np.hstack((-1.0, b_in, 1.0))
    if breaks is not None:
        assert np.array_equal(b_in, breaks)
    s = np.hstack((-1.0, tau))
    assert np.abs(D @ np.ones(n + 1)).max() <= 64 * EPS * np.abs(D).max()
    rng = np.random.default_rng(n)
    r = 0
    for k, (nk, c) in enumerate(zip(counts, cols)):
        assert tau[c + nk - 1] == b[k + 1]  # the interval's last node is its right end, exactly
        assert np.all(D[c:c + nk, :c] == 0.0) and np.all(D[c:c + nk, c + nk + 1:] == 0.0)
        w = b[k + 1] - b[k]
        assert _eq(D[c:c + nk, c:c + nk + 1], lgr_diff_matrix(nk, lgr_nodes(nk) if nk > 1 else np.ones(1)) * (2.0 / w))
        # exact, to rounding, on a polynomial of degree n_k over the interval
        coef = rng.normal(size=nk + 1)
        sk = s[c:c + nk + 1]
        want = np.polyval(np.polyder(coef), sk[1:])
        got = D[c:c + nk] @ np.polyval(coef, s)
        assert np.allclose(got, want, rtol=0, atol=1e-10 * np.abs(coef).sum() * (2.0 / w) ** nk), (k, got - want)
        r += nk
    # a section of one interval is today's, bit for bit
    for iv in (None, ([n], None), ([n], [])):
        one = PSparams([n], [iv])
        assert one.tau(0) is mesh_tables(n)[0] and one.D(0) is mesh_tables(n)[1]
        assert one.intervals(0)[0] == [n] and one.intervals(0)[2] == [0]


def test_interval_validation_and_event_records(tmp_path):
    for counts, breaks in (([8, 7], None), ([0, 16], None), ([8, 8], [0.0, 0.5]), ([8, 8], [1.0]), ([8, 8], [-1.0]),
                           ([4, 4, 8], [0.2, 0.1]), ([8, 8], [np.nan])):
        with pytest.raises(ValueError):
            PSparams([16], [(counts, breaks)])
    ev = helpers.example_inputs()["events"]
    for bad in ({"mesh_intervals": [8, 7]}, {"mesh_breaks": [0.0]}, {"mesh_intervals": [8, 8], "mesh_breaks": [2.0]}):
        e = dict(ev[2], **bad)
        with pytest.raises(ValueError, match="ZEROLIFT_START"):
            problem.event_intervals(e)
    # records without the keys build today's problem; the CSV columns are optional and ';'-separated
    inp = _with_intervals(helpers.example_inputs(), SPLITS["zl_3_unequal"])
    header = list(ev[0].keys())
    rows = []
    for e in inp["events"]:
        row = ["" if (isinstance(e[k], float) and e[k] != e[k]) else str(e[k]) for k in header]
        rows.append(row + [";".join(str(v) for v in e.get("mesh_intervals", [])),
                           ";".join(repr(v) for v in e.get("mesh_breaks", []))])
    path = tmp_path / "events.csv"
    path.write_text("\n".join(",".join(r) for r in [header + ["mesh_intervals", "mesh_breaks"]] + rows) + "\n")
    got = problem.read_events(str(path))
    assert [e.get("mesh_intervals") for e in got] == [e.get("mesh_intervals") for e in inp["events"]]
    assert [e.get("mesh_breaks") for e in got] == [e.get("mesh_breaks") for e in inp["events"]]
    plain = tmp_path / "plain.csv"
    plain.write_text("\n".join(",".join(r[:len(header)]) for r in [header] + rows) + "\n")
    assert all("mesh_intervals" not in e for e in problem.read_events(str(plain)))


@pytest.mark.parametrize("name", sorted(SPLITS))
@pytest.mark.parametrize("mode", ["forward", "central"])
def test_nlp_on_composite_meshes_equals_oracle_bit_for_bit(name, mode):
    inp, p, u, c, x0, O, P = _setup(name, mode)
    Lg = leaves.get("gmath")
    pp, up, cp, _ = problem.problem_from_inputs(_plain(inp), coord=Lg.coordinate_c)
    Pp = helpers.compiled_plan(pp, up, cp, coord=Lg.coordinate_c)
    assert (P.n_vars, P.n_rows, P.n_vals) == (Pp.n_vars, Pp.n_rows, Pp.n_vals)
    assert np.array_equal(P.xdep_index(), Pp.xdep_index())
    E, Ep = emu_binding.Emulator(P), emu_binding.Emulator(Pp)
    assert E.n_pack == Ep.n_pack
    E.set_fd(mode)
    keys = list(x0.keys())
    for x in (x0, helpers.perturbed(x0)):
        xv = problem.xdict_to_vector(x)
        f, _ = O.objfunc(helpers.copy_x(x))
        helpers.assert_funcs_equal(f, P.split_residuals(E.eval_residuals(xv)))
        s, _ = O.sens(helpers.copy_x(x))
        vals = E.eval_jacobian(xv)
        assert not np.isnan(vals).any()
        helpers.assert_sens_equal(s, P.split_jacobian(vals, key_order=keys))
        sp = Pp.split_jacobian(Ep.eval_jacobian(xv), key_order=keys)  # the same COO rows / columns
        for grp, blk in P.split_jacobian(vals, key_order=keys).items():
            for var, b in (blk or {}).items():
                if isinstance(b, dict):
                    assert np.array_equal(b["coo"][0], sp[grp][var]["coo"][0]) and \
                        np.array_equal(b["coo"][1], sp[grp][var]["coo"][1]), (grp, var)


def _grids(ps):
    return [mesh.grid_tables(ps), mesh.grid_tables(ps, m=3)]


@pytest.mark.parametrize("name", sorted(SPLITS))
def test_per_interval_estimate_equals_oracle_bit_for_bit(name):
    inp, p, u, c, x0, O, P = _setup(name)
    E = emu_intervals.IntervalEmuEngine(P)
    x_sol = mesh.transfer(_solution(), helpers.example_problem(coord=leaves.get("gmath").coordinate_c)[0]["ps_params"],
                          O.ps)
    for tabs in _grids(O.ps):
        assert "n_int" in tabs and tabs["int_m"].size == tabs["int_base"].size == sum(tabs["n_int"])
        E.set_mesh_grid(tabs)
        for x in (x0, helpers.perturbed(x0), x_sol):
            xv = problem.xdict_to_vector(x)
            wi, ws = mesh_intervals_oracle.mesh_error_intervals(O, x, tabs)
            gi, gs = E.mesh_error_intervals(xv), E.mesh_error(xv)
            assert _eq(gi, wi) and _eq(gs, ws)
            k = 0
            for i in range(O.S):  # the section's value is the max of its intervals
                K = int(tabs["n_int"][i])
                assert _eq(gs[i], gi[k:k + K].max(axis=0))
                k += K


def test_gelato_problem_mesh_error_intervals_on_the_emulator():
    from gelato_b200 import callbacks

    inp, p, u, c, x0, O, P = _setup("zl_3_unequal")
    Lg = leaves.get("gmath")
    prob = callbacks.GelatoProblem(p, u, c, user_eq=callbacks.PerigeeAtEvent(helpers.USER_EVENT), coord=Lg.coordinate_c,
                                   engine_factory=emu_intervals.IntervalEmuEngine)
    x = helpers.perturbed(x0)
    got, sec = prob.mesh_error_intervals(x), prob.mesh_error(x)
    wi, ws = mesh_intervals_oracle.mesh_error_intervals(O, x, mesh.grid_tables(p["ps_params"]))
    names = [e["name"] for e in p["params"][:-1]]
    assert list(got) == names and [len(got[k]) for k in names] == [len(p["ps_params"].intervals(i)[0]) for i in range(O.S)]
    assert _eq(np.concatenate([got[k] for k in names]), wi) and _eq(np.stack([sec[k] for k in names]), ws)
    prob.close()


def test_single_interval_grids_are_todays():
    _, p, u, c, x0, O, P = _setup("zl_8_8")
    ps = helpers.example_problem()[0]["ps_params"]
    t = mesh.grid_tables(ps)
    assert set(t) == {"m", "off", "pool"}
    for i in range(ps.num_sections()):
        for a, b in zip(mesh_oracle.unpack(t, i, ps.nodes(i)), mesh.section_tables(ps.tau(i), ps.nodes(i) + 1)):
            assert _eq(a, b)
    with pytest.raises(ValueError):
        mesh.grid_tables(O.ps, m=[3] * O.S)  # a per-section list needs single-interval sections


def test_square_grid_identity_per_interval():
    """m_k = n_k test points per interval (the interval's own nodes): the estimate of interval k is
    |w_k / 2 A_k^-1 g_k| / scale on the D.X rows (g_k its collocation defects) and |X_l - X_base| / scale on the
    difference rows."""
    _, p, u, c, x0, O, P = _setup("coast")
    x = helpers.perturbed(x0)
    ps = O.ps
    parts, off, o, ims = [], [], 0, []
    for i in range(O.S):
        counts, breaks, cols = ps.intervals(i)
        tt, Pm, Qm, I = mesh.interval_tables(ps.tau(i), counts, breaks, counts) if len(counts) > 1 else \
            mesh.section_tables(ps.tau(i), counts[0])
        off.append(o)
        for a in (tt, Pm, Qm, I):
            parts.append(a.ravel())
            o += a.size
        ims += counts
    tabs = {"m": np.array([ps.nodes(i) for i in range(O.S)], dtype=np.int32), "off": np.array(off, dtype=np.int64),
            "pool": np.concatenate(parts), "n_int": np.array([len(ps.intervals(i)[0]) for i in range(O.S)], dtype=np.int32),
            "int_m": np.array(ims, dtype=np.int32),
            "int_base": np.array([cc for i in range(O.S) for cc in ps.intervals(i)[2]], dtype=np.int32)}
    E = emu_intervals.IntervalEmuEngine(P)
    E.set_mesh_grid(tabs)
    err = E.mesh_error_intervals(problem.xdict_to_vector(x))
    g, _ = O.objfunc(helpers.copy_x(x))
    dyn = np.column_stack((g["eqcon_dyn_mass"], g["eqcon_dyn_pos"].reshape(-1, 3), g["eqcon_dyn_vel"].reshape(-1, 3),
                           g["eqcon_dyn_quat"].reshape(-1, 4)))
    r = 0
    for i in range(O.S):
        ua, ub, xa, xb, n = ps.get_index(i)
        counts, breaks, cols = ps.intervals(i)
        b = np.hstack((-1.0, breaks, 1.0))
        X, _ = mesh_oracle.section_states(O, x, i)
        diff_rows = [0] * (not O.p["params"][i]["engineOn"]) + [7, 8, 9, 10] * O._holds(i)
        for k, (nk, cc) in enumerate(zip(counts, cols)):
            Xk = X[cc:cc + nk + 1]
            scale = 1.0 + np.max(np.abs(Xk[1:]), axis=0)
            A = lgr_diff_matrix(nk, lgr_nodes(nk) if nk > 1 else np.ones(1))[:, 1:]
            gk = dyn[ua + cc:ua + cc + nk]
            for comp in range(11):
                if comp in diff_rows:
                    want = np.max(np.abs(Xk[1:, comp] - Xk[0, comp])) / scale[comp]
                    assert err[r, comp] == want, (i, k, comp)
                    continue
                want = np.max(np.abs(np.linalg.solve(A, gk[:, comp]) * ((b[k + 1] - b[k]) / 2.0))) / scale[comp]
                bound = 1e-12 * (1.0 + np.max(np.abs(Xk[:, comp]))) * np.abs(np.linalg.inv(A)).sum(axis=1).max() / scale[comp]
                assert abs(err[r, comp] - want) <= bound + 1e-9 * want, (i, k, comp, err[r, comp], want)
            r += 1


# Largest component estimate of the section at n nodes per interval, K = 1, 2, 4 intervals (DOP853 state), and the
# ratio of each halving of the interval width (order n + 1: 8 for n = 2, 16 for n = 3):
#   SECO n = 2  1.02e-06  1.33e-07  1.69e-08   7.7  7.9
#   SECO n = 3  8.53e-10  5.35e-11  3.35e-12  15.9 16.0
#   SEP2 n = 2  1.01e-09  1.27e-10  1.59e-11   8.0  8.0
#   SEP2 n = 3  8.57e-14  5.30e-15  3.41e-16  16.2 15.6
@pytest.mark.parametrize("event", ["SECO", "SEP2"])
@pytest.mark.parametrize("n", [2, 3])
def test_vacuum_coast_estimate_falls_with_intervals(event, n):
    Lg = leaves.get("gmath")
    ps0 = helpers.example_problem(coord=Lg.coordinate_c)[0]["ps_params"]
    x_sol = _solution()
    errs = []
    for K in (1, 2, 4):
        def mutate(inp, K=K):
            for e in inp["events"]:
                if e["name"] == event:
                    e["num_nodes"] = n * K
                    if K > 1:
                        e["mesh_intervals"] = [n] * K

        p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c, mutate=mutate)
        i = p["event_index"][event]
        O = helpers.oracle_nlp(p, u, c, "gmath", "seqfma")
        x = _coast_state(O, mesh.transfer(x_sol, ps0, O.ps), i)
        ei, _ = mesh_intervals_oracle.mesh_error_intervals(O, x, mesh.grid_tables(O.ps))
        k0 = sum(len(O.ps.intervals(j)[0]) for j in range(i))
        errs.append(float(ei[k0:k0 + K].max()))
    floor = 1e-12
    for a, b in zip(errs, errs[1:]):
        assert b < a / 4.0 or max(a, b) < floor, errs


def _malformed(tabs):
    """(grid, why) copies of a composite grid with one interval defect each (plan_host.h: build_mesh_grid)."""
    out = []
    for key, i, value, why in (("n_int", 2, 0, "at least one interval"),
                               ("int_m", 3, 1, "do not add up"),
                               ("int_m", 3, 0, "do not add up"),
                               ("int_base", 3, 0, "base column"),
                               ("int_base", 2, 1, "base column"),
                               ("int_base", 3, 99, "base column")):
        t = {k: v.copy() for k, v in tabs.items()}
        t[key][i] = value
        out.append((t, why))
    return out


def test_grid_refusals_keep_the_previous_grid():
    _, p, u, c, x0, O, P = _setup("zl_3_unequal")
    E = emu_intervals.IntervalEmuEngine(P)
    x = problem.xdict_to_vector(helpers.perturbed(x0))
    tabs = mesh.grid_tables(O.ps)
    assert list(tabs["n_int"][:4]) == [1, 1, 3, 1]  # intervals of section 2 at indices 2, 3, 4
    E.set_mesh_grid(tabs)
    ref, ref_i = E.mesh_error(x), E.mesh_error_intervals(x)
    for t, why in _malformed(tabs):
        with pytest.raises(engine.GelatoError, match="gelato_plan_set_mesh_grid.*" + why):
            E.set_mesh_grid(t)
        assert _eq(E.mesh_error(x), ref) and _eq(E.mesh_error_intervals(x), ref_i)
    with pytest.raises(engine.GelatoError, match="at least one interval"):
        t = {k: v.copy() for k, v in tabs.items()}
        t["n_int"][0] = -1
        E.set_mesh_grid(t)
    # the same grid without interval tables: one interval per section (per-section values unchanged where K = 1)
    plain = {k: tabs[k] for k in ("m", "off", "pool")}
    E.set_mesh_grid(plain)
    assert E.mesh_error_intervals(x).shape == (O.S, 11)


def _events(splits=None):
    ev = helpers.example_inputs()["events"]
    return _with_intervals({"events": ev, "settings": {}}, splits or {})["events"]


def test_refine_nodes_ph_rule():
    ev = _events({"ZEROLIFT_START": ([8, 8], None)})
    S = len(ev) - 1
    K = [len(e.get("mesh_intervals", [1])) for e in ev[:S]]
    err = np.zeros((sum(K), 11))
    # rows: LIFTOFF 0, KICKTURN 1, ZEROLIFT_START 2 and 3, ZEROLIFT_END 4, ...
    err[0, 3] = 1e-3   # n = 5: 5 + ceil(log(1e3) / log(5)) = 10 <= 12: p branch
    err[3, 1] = 1e-2   # ZEROLIFT_START's second interval, n = 8: 8 + 5 = 13 > 12: split into ceil(13 / 4) = 4 x 4
    err[4, 0] = 1e-1   # ZEROLIFT_END, n = 8: 8 + 7 = 15 > 12: split into 4 x 4
    new, rep = mesh.refine_nodes(ev, err, tol=1e-6, n_max=12, n_min=4)
    got = {(r.name, r.interval): (r.n_old, r.n_new, r.split, r.capped) for r in rep}
    assert got[("LIFTOFF", 0)] == (5, 10, 1, False)
    assert got[("ZEROLIFT_START", 0)] == (8, 8, 1, False)
    assert got[("ZEROLIFT_START", 1)] == (8, 16, 4, False)
    assert got[("ZEROLIFT_END", 0)] == (8, 16, 4, False)
    zs, ze = new[2], new[3]
    assert zs["mesh_intervals"] == [8, 4, 4, 4, 4] and zs["num_nodes"] == 24
    assert zs["mesh_breaks"] == [0.0, 0.25, 0.5, 0.75]
    assert ze["mesh_intervals"] == [4, 4, 4, 4] and ze["mesh_breaks"] == [-0.5, 0.0, 0.5]
    assert "mesh_intervals" not in new[0] and new[0]["num_nodes"] == 10
    # the new events build, and the same errors without n_min cap as before
    PSparams([e["num_nodes"] for e in new[:S]], [problem.event_intervals(e) for e in new[:S]])
    _, rep2 = mesh.refine_nodes(ev, err, tol=1e-6, n_max=12)
    assert [(r.n_new, r.capped) for r in rep2 if r.name == "ZEROLIFT_END"] == [(12, True)]
    # the dictionary form of GelatoProblem.mesh_error_intervals gives the same result
    d, k = {}, 0
    for i, e in enumerate(ev[:S]):
        d[e["name"]] = err[k:k + K[i]]
        k += K[i]
    assert mesh.refine_nodes(ev, d, tol=1e-6, n_max=12, n_min=4) == (new, rep)
    with pytest.raises(ValueError):
        mesh.refine_nodes(ev, np.zeros((S, 11)), tol=1e-6, n_max=12)  # a section of 2 intervals needs 2 estimates


def test_refine_nodes_path_drives_the_interval_of_the_worst_residual():
    ev = _events({"ZEROLIFT_START": ([8, 8], [0.5])})
    S = len(ev) - 1
    err = np.zeros((S + 1, 11))
    to, tf = ev[2]["time"], ev[3]["time"]
    t_at = lambda tau: (tau + 1.0) * (tf - to) / 2.0 + to  # noqa: E731
    path = {("ineqcon_qalpha", "ZEROLIFT_START"): (-4e-3, t_at(0.7)), ("ineqcon_alpha", "ZEROLIFT_START"): (0.1, t_at(0.0)),
            ("ineqcon_alpha", "LIFTOFF"): (0.2, ev[0]["time"])}
    new, rep = mesh.refine_nodes(ev, err, tol=1e-6, n_max=12, path=path, path_tol=1e-3, n_min=4)
    zs = [r for r in rep if r.name == "ZEROLIFT_START"]
    assert [(r.interval, r.n_new, r.path) for r in zs] == [(0, 8, None), (1, 8 + 1, -4e-3)]  # tau 0.7 > break 0.5
    assert new[2]["mesh_intervals"] == [8, 9]
    # a residual on the breakpoint drives the interval on its left
    path[("ineqcon_qalpha", "ZEROLIFT_START")] = (-4e-3, t_at(0.5))
    _, rep = mesh.refine_nodes(ev, err, tol=1e-6, n_max=12, path=path, n_min=4)
    assert [(r.interval, r.path) for r in rep if r.name == "ZEROLIFT_START"] == [(0, -4e-3), (1, None)]
    # single-interval events without n_min: today's report (one Refinement per section, interval 0, split 1)
    ev1 = _events()
    new1, rep1 = mesh.refine_nodes(ev1, np.full((S, 11), 1e-3), tol=1e-6, n_max=40)
    assert all(r.interval == 0 and r.split == 1 for r in rep1) and all("mesh_intervals" not in e for e in new1)


def _poly_x(ps, rng):
    """a decision vector whose states are continuous polynomials of degree n_k and controls polynomials of degree
    n_k - 1 per interval; (x, coefficients)"""
    M, N = ps.num_x(), ps.num_u()
    x = {"mass": np.empty(M), "position": np.empty(3 * M), "velocity": np.empty(3 * M), "quaternion": np.empty(4 * M),
         "u": np.empty(2 * N), "t": np.linspace(0.0, 0.5, ps.num_sections() + 1)}
    coef = {}
    for i in range(ps.num_sections()):
        ua, ub, xa, xb, n = ps.get_index(i)
        counts, breaks, cols = ps.intervals(i)
        s = np.hstack((-1.0, ps.tau(i)))
        b = np.hstack((-1.0, breaks, 1.0))
        for k, (nk, c) in enumerate(zip(counts, cols)):
            for key, w in (("mass", 1), ("position", 3), ("velocity", 3), ("quaternion", 4), ("u", 2)):
                cf = rng.normal(size=(w, nk if key == "u" else nk + 1))
                if key != "u" and k > 0:  # continuous states: the interval starts where the previous one ends
                    prev = coef[i, k - 1, key][0]
                    cf[:, -1] += [np.polyval(prev[j], b[k]) - np.polyval(cf[j], b[k]) for j in range(w)]
                coef[i, k, key] = (cf, b[k], b[k + 1])
                pts = ps.tau(i)[c:c + nk] if key == "u" else s[c + (k > 0):c + nk + 1]
                first = (ua + c) if key == "u" else (xa + c + (k > 0))
                x[key].reshape(-1, w)[first:first + pts.size] = np.stack([np.polyval(cf[j], pts) for j in range(w)], axis=1)
    return x, coef


def test_transfer_reproduces_piecewise_polynomials():
    rng = np.random.default_rng(5)
    # section 1 of the old mesh is one interval, section 2 is split; the new mesh splits 1 and refines 2; 0 is unchanged
    ps = PSparams([3, 4, 6], [None, None, ([3, 3], [0.2])])
    ps2 = PSparams([3, 9, 10], [None, ([4, 5], [-0.3]), ([3, 2, 3, 2], [-0.4, 0.2, 0.6])])
    x, coef = _poly_x(ps, rng)
    y = mesh.transfer(x, ps, ps2)
    assert list(y) == list(x) and _eq(y["t"], x["t"])
    for i in (1, 2):
        ua, ub, xa, xb, n = ps2.get_index(i)
        s2 = np.hstack((-1.0, ps2.tau(i)))
        counts, breaks, cols = ps.intervals(i)
        b = np.hstack((-1.0, breaks, 1.0))
        for r, t in enumerate(s2):
            k = min(int(np.searchsorted(b[1:-1], t, side="left")), len(counts) - 1)
            for key, w in (("mass", 1), ("position", 3), ("velocity", 3), ("quaternion", 4)):
                cf = coef[i, k, key][0]
                want = np.array([np.polyval(cf[j], t) for j in range(w)])
                assert np.allclose(y[key].reshape(-1, w)[xa + r], want, rtol=0, atol=1e-11 * np.abs(cf).sum())
            if r > 0:
                cf = coef[i, k, "u"][0]
                want = np.array([np.polyval(cf[j], t) for j in range(2)])
                assert np.allclose(y["u"].reshape(-1, 2)[ua + r - 1], want, rtol=0, atol=1e-11 * np.abs(cf).sum())
    # the breakpoint 0.2 of the old section 2 is a node of the new one: copied from the old node there
    xa_old = ps.get_index(2)[2]
    xa_new = ps2.get_index(2)[2]
    j_old = 1 + int(np.nonzero(ps.tau(2) == 0.2)[0][0])
    j_new = 1 + int(np.nonzero(ps2.tau(2) == 0.2)[0][0])
    assert _eq(y["position"].reshape(-1, 3)[xa_new + j_new], x["position"].reshape(-1, 3)[xa_old + j_old])
    # unchanged section: bit for bit; the same mesh: every key bit for bit
    assert _eq(y["velocity"].reshape(-1, 3)[0:4], x["velocity"].reshape(-1, 3)[0:4])
    same = mesh.transfer(x, ps, ps)
    assert all(_eq(same[k], x[k]) for k in x)


@pytest.mark.parametrize("name", ["zl_8_8", "zl_3_unequal"])
def test_path_check_and_path_rows_on_composite_grids(name):
    inp, p, u, c, x0, O, P = _setup(name)
    E = emu_binding.EmuEngine(P)
    i = p["event_index"]["ZEROLIFT_START"]
    for tabs in _grids(O.ps):
        E.set_mesh_grid(tabs)
        E.set_path_rows(tabs)
        lay = E.path_rows_layout()
        jobs = {(int(k), int(s)): j for j, (k, s, nk, _) in enumerate(P.aero_i32)}
        want_rows = [(jobs[(path_rows_oracle.KINDS.index(kind), s)], l)
                     for kind, s, _, l in path_rows_oracle.row_list(O, tabs)]
        assert list(zip(lay["job"], lay["l"])) == want_rows
        # test points on the interior breakpoints have unit P rows and carry no row
        tau_t, Pm, _, _ = mesh_oracle.unpack(tabs, i, O.ps.nodes(i))
        on_break = [l for l in range(tau_t.size) if tau_t[l] in set(O.ps.intervals(i)[1])]
        assert len(on_break) == len(O.ps.intervals(i)[1])
        for l in on_break:
            assert np.count_nonzero(Pm[l]) == 1 and Pm[l].max() == 1.0
            assert all(ll != l for j, ll in zip(lay["job"], lay["l"]) if P.aero_i32[j][1] == i)
        for mode in ("forward", "central"):
            E.set_fd(mode)
            for x in (x0, helpers.perturbed(x0)):
                xv = problem.xdict_to_vector(x)
                res, at = E.path_check(xv)
                wr, wa = path_oracle.path_check(O, x, tabs)
                assert _eq(res, wr) and np.array_equal(at, wa)
                g, v = E.eval_path_rows(xv)
                gw, vw = path_rows_oracle.path_rows(O, x, tabs, mode)
                assert _eq(g, gw) and _eq(v, vw)
        # the P-weighted entries of a row in section i are explicit zeros outside its interval
        E.set_fd("forward")
        _, v = E.eval_path_rows(problem.xdict_to_vector(helpers.perturbed(x0)))
        n = O.ps.nodes(i)
        for r, (j, l) in enumerate(zip(lay["job"], lay["l"])):
            if P.aero_i32[j][1] != i:
                continue
            ent = v[lay["off"][r][0]:lay["off"][r][0] + 3 * (n + 1)].reshape(n + 1, 3)
            zero = Pm[l] == 0.0
            assert zero.any() and np.all(ent[zero] == 0.0) and np.any(ent[~zero] != 0.0)


def test_host_users_of_tau():
    inp, p, u, c, x0, O, P = _setup("zl_3_unequal")
    pp = problem.problem_from_inputs(_plain(inp))[0]
    ps = p["ps_params"]
    tc, tx = problem.section_time_grids(p)
    i = p["event_index"]["ZEROLIFT_START"]
    to, tf = p["params"][i]["time"], p["params"][i]["timeFinishAt"]
    ua, ub, xa, xb, n = ps.get_index(i)
    assert np.array_equal(tc[ua:ub], ps.tau(i) * (tf - to) / 2.0 + (tf + to) / 2.0)
    assert np.all(np.diff(tx[xa:xb]) > 0) and tx[xa] == to
    # the breakpoints are node times
    for bk in ps.intervals(i)[1]:
        assert np.any(tc[ua:ub] == bk * (tf - to) / 2.0 + (tf + to) / 2.0)
    tn, txn = initialize.mesh_times(p)
    assert np.array_equal(tn, tc) and np.array_equal(txn, tx)
    # the initial guess follows the composite node times, the layout is that of the same node counts
    assert all(x0[k].shape == problem.problem_from_inputs(_plain(inp))[3][k].shape for k in x0)
    assert not np.array_equal(x0["position"], problem.problem_from_inputs(_plain(inp))[3]["position"])
    sec, event, _ = output.row_sections(p, p["M"])
    assert np.array_equal(sec, output.row_sections(pp, pp["M"])[0])

    class _Prob:
        pass

    st = nlpshim.attach_structure(_Prob(), p).structure
    assert st == nlpshim.attach_structure(_Prob(), pp).structure


def _solution():
    Lg = leaves.get("gmath")
    P = helpers.compiled_plan(*helpers.example_problem(coord=Lg.coordinate_c)[:3], coord=Lg.coordinate_c)
    x = np.load(helpers.GOLDEN + "/example_solution.npz")["x"]
    return problem.vector_to_xdict(x, P.M, P.N, P.S)


# ------------------------------------------------------------------------------------------------ GPU tier
def _engine(P, scenario_plans=None):
    return engine.Engine(P, device=0, scenario_plans=scenario_plans)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SPLITS))
@pytest.mark.parametrize("mode", ["forward", "central"])
def test_gpu_nlp_on_composite_meshes(name, mode):
    inp, p, u, c, x0, O, P = _setup(name, mode)
    E = _engine(P)
    E.set_fd(mode)
    Em = emu_binding.Emulator(P)
    Em.set_fd(mode)
    keys = list(x0.keys())
    full, src, sgn = Em.packed_map()
    for x in (x0, helpers.perturbed(x0)):
        xv = problem.xdict_to_vector(x)
        f, _ = O.objfunc(helpers.copy_x(x))
        g = E.eval_residuals(xv)
        helpers.assert_funcs_equal(f, P.split_residuals(g))
        s, _ = O.sens(helpers.copy_x(x))
        vals = E.eval_jacobian(xv)
        helpers.assert_sens_equal(s, P.split_jacobian(vals, key_order=keys))
        # pair, packed and update modes
        gp, pk = np.empty(P.n_rows), np.empty(E.L.gelato_plan_n_pack(E.h))
        assert E.L.gelato_eval_pair_packed(E.h, xv.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                           gp.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                           pk.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), 1) == 0
        assert _eq(gp, g)
        v = P.vals_template.copy()
        v[full] = sgn * pk[src]
        assert _eq(v, vals)
        buf_g, buf_v = np.empty(P.n_rows), np.empty(P.n_vals)
        E.jacobian_template(buf_v)
        E.eval_pair_update(xv, buf_g, buf_v)
        assert _eq(buf_g, g) and _eq(buf_v, vals)
    E.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SPLITS))
def test_gpu_per_interval_estimate_equals_oracle(name):
    inp, p, u, c, x0, O, P = _setup(name)
    E = _engine(P)
    for tabs in _grids(O.ps):
        E.set_mesh_grid(tabs)
        for x in (x0, helpers.perturbed(x0)):
            xv = problem.xdict_to_vector(x)
            wi, ws = mesh_intervals_oracle.mesh_error_intervals(O, x, tabs)
            assert _eq(E.mesh_error_intervals(xv), wi) and _eq(E.mesh_error(xv), ws)
    E.close()


@pytest.mark.gpu
def test_gpu_dispersed_batch_and_buffers():
    import torch

    Lg = leaves.get("gmath")
    base = _with_intervals(helpers.example_inputs(), SPLITS["zl_3_unequal"])
    scen = scenarios.disperse(base, 64, seed=11)
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
    err = E.mesh_error_intervals(X, n_scen=64)
    sec = E.mesh_error(X, n_scen=64)
    for k in range(64):
        wi, ws = mesh_intervals_oracle.mesh_error_intervals(oracles[k], xs[k], tabs)
        assert _eq(err[k], wi) and _eq(sec[k], ws), k
    assert not _eq(err[0], err[1])
    # pinned host buffers and device pointers
    px, pe = engine.PinnedArray(X[:3].size), engine.PinnedArray(err[:3].size)
    px.array[:] = X[:3].ravel()
    E.mesh_error_intervals(px.array, n_scen=3, out=pe.array)
    assert _eq(pe.array.reshape(err[:3].shape), err[:3])
    xd = torch.from_numpy(X[:3].copy()).cuda()
    ed = torch.full(err[:3].shape, float("nan"), dtype=torch.float64, device="cuda")
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        E.mesh_error_intervals_dev(xd.data_ptr(), ed.data_ptr(), 3, st.cuda_stream)
    st.synchronize()
    assert _eq(ed.cpu().numpy(), err[:3])
    assert _eq(E.mesh_error_intervals(X[0]), err[0])  # a smaller batch after a larger one (scenario 0's blocks)
    px.free()
    pe.free()
    E.close()


@pytest.mark.gpu
def test_gpu_bench_workload_sample_with_two_sections_split():
    import bench

    Lg = leaves.get("gmath")
    scen = scenarios.disperse(bench.workload_inputs("example"), 128, seed=20260117)
    plans, X, probs = [], [], []
    for k in range(128):
        inp = _with_intervals(scen[k], {"ZEROLIFT_START": ([10, 10], None), "ZEROLIFT_START__1": ([7, 7, 6], [-0.5, 0.25])},
                              factor=15)
        p, u, c, x0 = problem.problem_from_inputs(inp, coord=Lg.coordinate_c)
        rng = np.random.default_rng(1000 + k)
        x = {key: v + (0.0 if key == "t" else 1e-3) * rng.uniform(-1.0, 1.0, v.shape) for key, v in x0.items()}
        plans.append(helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c))
        X.append(problem.xdict_to_vector(x))
        probs.append((p, u, c, x))
    X = np.stack(X)
    assert sum(len(plans[0].ps.intervals(i)[0]) > 1 for i in range(plans[0].S)) == 2
    E = _engine(plans[0], scenario_plans=plans)
    tabs = mesh.grid_tables(plans[0].ps)
    E.set_mesh_grid(tabs)
    err = E.mesh_error_intervals(X, n_scen=128)
    g = E.eval_residuals(X, n_scen=128)
    assert err.shape == (128, int(tabs["n_int"].sum()), 11) and np.isfinite(err).all()
    for k in (0, 37, 127):
        p, u, c, x = probs[k]
        O = helpers.oracle_nlp(p, u, c, "gmath", "seqfma")
        wi, ws = mesh_intervals_oracle.mesh_error_intervals(O, x, tabs)
        assert _eq(err[k], wi), k
        f, _ = O.objfunc(helpers.copy_x(x))
        helpers.assert_funcs_equal(f, plans[k].split_residuals(g[k]))
    E.close()


@pytest.mark.gpu
def test_gpu_grid_refusals_keep_the_previous_grid():
    _, p, u, c, x0, O, P = _setup("zl_3_unequal")
    E = _engine(P)
    x = problem.xdict_to_vector(helpers.perturbed(x0))
    tabs = mesh.grid_tables(O.ps)
    E.set_mesh_grid(tabs)
    ref, ref_i = E.mesh_error(x), E.mesh_error_intervals(x)
    for t, why in _malformed(tabs):
        with pytest.raises(engine.GelatoError, match="gelato_plan_set_mesh_grid.*" + why):
            E.set_mesh_grid(t)
        assert _eq(E.mesh_error(x), ref) and _eq(E.mesh_error_intervals(x), ref_i)
    err = np.empty(O.S * 11)
    assert E.L.gelato_eval_mesh_error_intervals(E.h, x.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), None, 1) == -1
    assert E.L.gelato_eval_mesh_error_intervals(E.h, x.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                                err.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), 0) == -1
    E.close()
