"""GPU tier: the host side of a plan -- the per-scenario blocks of gelato_plan_set_scenarios and the staging buffers
that every host-buffer entry point shares -- checked bit for bit against fresh plans and the device-pointer entry
points."""
import ctypes

import numpy as np
import pytest

import helpers
from gelato_b200 import engine, problem, scenarios
from oracle import leaves

pytestmark = pytest.mark.gpu


def _plans(n, factor=1, seed=3):
    """The nominal example plan and n dispersed scenarios of it (none nominal), with a perturbed x for each."""
    Lg = leaves.get("gmath")
    plans, xs = [], []
    for si in scenarios.disperse(helpers.example_inputs(), n + 1, seed=seed):
        p, u, c, x0 = problem.problem_from_inputs(si, coord=Lg.coordinate_c, factor=factor)
        plans.append(helpers.compiled_plan(p, u, c, coord=Lg.coordinate_c))
        xs.append(problem.xdict_to_vector(helpers.perturbed(x0, seed=len(xs))))
    return plans[0], plans[1:], np.stack(xs[1:])


def test_null_scenario_member_means_the_shared_block_after_an_earlier_call():
    """A NULL member of GelatoScenarioDesc is the block every scenario shares, whatever an earlier call configured:
    all five blocks, then only sec_f64, evaluates like a fresh plan given only the second call."""
    base, plans, X = _plans(6)
    first, second, X = plans[:3], plans[3:], X[:3]
    assert all(not np.array_equal(p.wind, base.wind) for p in first)
    assert all(not np.array_equal(p.vals_template, base.vals_template) for p in first)

    def set_scenarios(E, scen_plans, only_sec_f64):
        sc, keep = engine.make_scenario_desc(scen_plans)
        if only_sec_f64:
            sc.wind = sc.unit_mass = sc.lin_const = sc.vals_template = None
        assert E.L.gelato_plan_set_scenarios(E.h, ctypes.byref(sc)) == 0, E.L.gelato_last_error()

    def results(E):
        g, pk = E.eval_pair_packed(X, 3)
        return E.eval_residuals(X, 3).copy(), E.eval_jacobian(X, 3).copy(), g.copy(), pk.copy()

    fresh = engine.Engine(base)
    set_scenarios(fresh, second, True)
    want = results(fresh)
    E = engine.Engine(base)
    set_scenarios(E, first, False)
    configured = results(E)
    assert not any(np.array_equal(a, b) for a, b in zip(configured, want))  # the first call's blocks do matter
    set_scenarios(E, second, True)
    for got, w in zip(results(E), want):
        assert np.array_equal(got, w)
    E.close()
    fresh.close()


def test_host_entry_points_share_their_staging():
    """x, g and scenario-id staging is shared by every host-buffer entry point.  Interleave the small objfunc call of
    the captured graph, a packed pair call on a larger batch (which grows the staging the graph baked in), the small
    call again, _ids calls and a sliced update-mode pair call, through pageable and page-locked buffers: every result
    equals the device-pointer entry points on the same x, bit for bit."""
    import torch

    n = 8
    base, plans, X = _plans(n, factor=2, seed=5)
    E = engine.Engine(plans[0], scenario_plans=plans)
    P = plans[0]
    assert (P.n_vars + P.n_rows) * 8 <= 64 * 1024  # one scenario takes the graph path
    assert n * P.n_vals * 8 > 512 * 1024  # the update-mode call takes the sliced path
    E.set_update_slices(3)
    full = P.xdep_index()

    def device(Xb):
        """(g, COO vals, packed) of batch slot k = scenario k, through the device-pointer entry points."""
        m = Xb.shape[0]
        xd = torch.from_numpy(np.ascontiguousarray(Xb)).cuda()
        gd = [torch.full((m, P.n_rows), float("nan"), dtype=torch.float64, device="cuda") for _ in range(3)]
        vd = torch.empty((m, P.n_vals), dtype=torch.float64, device="cuda")
        pd = torch.full((m, E.n_pack), float("nan"), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        E.eval_residuals_dev(xd.data_ptr(), gd[0].data_ptr(), m)
        E.fill_template(vd.data_ptr(), m)
        E.eval_pair_dev(xd.data_ptr(), gd[1].data_ptr(), vd.data_ptr(), m)
        E.eval_pair_packed_dev(xd.data_ptr(), gd[2].data_ptr(), pd.data_ptr(), m)
        torch.cuda.synchronize()
        g = [t.cpu().numpy() for t in gd]
        assert np.array_equal(g[0], g[1]) and np.array_equal(g[0], g[2])
        return g[0], vd.cpu().numpy(), pd.cpu().numpy()

    g_want, v_want, pk_want = device(X)
    assert len({v_want[k].tobytes() for k in range(n)}) == n  # the scenarios do differ
    ids = np.array([6, 1, 4], dtype=np.int32)
    for pinned in (False, True):
        held = []

        def buf(m):
            if not pinned:
                return np.full(m, np.nan)
            held.append(engine.PinnedArray(m))
            held[-1].array[:] = np.nan
            return held[-1].array

        x1, g1, xn, gn, pkn, vn = (buf(m) for m in (P.n_vars, P.n_rows, X.size, n * P.n_rows, n * E.n_pack, n * P.n_vals))
        x1[:] = X[0]
        xn[:] = X.ravel()
        assert np.array_equal(E.eval_residuals(x1, 1, out=g1), g_want[0])
        G, PK = E.eval_pair_packed(xn, n, g_out=gn, packed_out=pkn)
        assert np.array_equal(G, g_want) and np.array_equal(PK, pk_want)
        g1[:] = np.nan
        assert np.array_equal(E.eval_residuals(x1, 1, out=g1), g_want[0])
        # batch slot j evaluates scenario ids[j] at X[ids[j]]
        xi = np.ascontiguousarray(X[ids])
        assert np.array_equal(E.eval_jacobian(xi, 3, scen_ids=ids), v_want[ids])
        G, PK = E.eval_pair_packed(xi, 3, scen_ids=ids)
        assert np.array_equal(G, g_want[ids]) and np.array_equal(PK, pk_want[ids])
        E.jacobian_template(vn, n)
        vn.reshape(n, -1)[:, full] = np.nan
        gn[:] = np.nan
        G, V = E.eval_pair_update(xn, gn, vn, n)
        assert np.array_equal(G, g_want) and np.array_equal(V, v_want), pinned
        for h in held:
            h.free()
    E.close()
