"""Pins the CPU oracle (oracle/) -- the checker every parity test relies on.

1. against the committed golden fixtures, which were produced by the REFERENCE'S
   OWN Python layer (tests/golden/make_golden.py);
2. live against that layer wherever /root/reference exists, on the shipped
   example and on variants that reach the constraint branches the example
   leaves cold (max-q, waypoint lat/lon/IIP rows, inclination, Fuel mode ...).
"""
import os

import numpy as np
import pytest

import helpers
import refharness
from gelato_b200 import problem
from oracle import leaves

GOLD_REF = os.path.join(helpers.GOLDEN, "example_reference.npz")
GOLD_GM = os.path.join(helpers.GOLDEN, "example_gmath.npz")


def _check_against_npz(npz, name, f, s, exact):
    """`exact`: bit-for-bit (gmath flavour is machine-independent).  Otherwise the
    libm flavour is allowed the last-bit freedom glibc's CPU-specific sin/cos/pow
    variants have, amplified by 1/dx in finite-difference slots (DESIGN.md H1)."""
    ff = helpers.flatten_funcs(f)
    assert sorted(k for k, v in f.items() if v is None) == sorted(npz["%s/none_f" % name].tolist())
    for k, v in ff.items():
        ref = npz["%s/f/%s" % (name, k)]
        assert v.shape == ref.shape, k
        if exact:
            assert np.array_equal(v, ref), k
        else:
            np.testing.assert_allclose(v, ref, rtol=0, atol=1e-13, err_msg=k)
    fs = helpers.flatten_sens(s)
    assert sorted(k for k, v in s.items() if v is None) == sorted(npz["%s/none_j" % name].tolist())
    n_blocks = len([k for k in npz.files if k.startswith(name + "/j/") and k.endswith("/data")])
    assert n_blocks == len(fs)
    for k, (r, c, d, shape) in fs.items():
        assert tuple(npz["%s/j/%s/shape" % (name, k)].tolist()) == tuple(shape), k
        if r is not None:
            assert r.dtype == np.int32 and c.dtype == np.int32
            assert np.array_equal(r, npz["%s/j/%s/rows" % (name, k)]), k
            assert np.array_equal(c, npz["%s/j/%s/cols" % (name, k)]), k
        ref = npz["%s/j/%s/data" % (name, k)]
        if exact:
            assert np.array_equal(d, ref), k
        else:
            np.testing.assert_allclose(d, ref, rtol=1e-9, atol=1e-6, err_msg=k)


@pytest.mark.parametrize("name", ["x0", "x1"])
def test_oracle_libm_matches_reference_golden(name):
    npz = np.load(GOLD_REF)
    p, u, c, x0 = helpers.example_problem()
    O = helpers.oracle_nlp(p, u, c, "libm", "numpy")
    x = problem.vector_to_xdict(npz["%s/x" % name].copy(), p["M"], p["N"], p["num_sections"])
    f, fail = O.objfunc(x)
    assert fail is False
    s, fail = O.sens(x)
    _check_against_npz(npz, name, f, s, exact=False)


def test_oracle_libm_matches_reference_golden_at_the_bench_workload():
    """The same at the workload bench.py times (example x15 in sections of <= 20 nodes, N = 990): the reference's
    own outputs in tests/golden/bench_reference.npz."""
    npz = np.load(os.path.join(helpers.GOLDEN, "bench_reference.npz"))
    p, u, c, x0 = helpers.example_problem(factor=15, max_nodes=20)
    O = helpers.oracle_nlp(p, u, c, "libm", "numpy")
    x = problem.vector_to_xdict(npz["x1/x"].copy(), p["M"], p["N"], p["num_sections"])
    f, fail = O.objfunc(x)
    assert fail is False
    s, fail = O.sens(x)
    _check_against_npz(npz, "x1", f, s, exact=False)


@pytest.mark.parametrize("name", ["x0", "x1"])
def test_oracle_gmath_matches_golden_bitwise(name):
    npz = np.load(GOLD_GM)
    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    O = helpers.oracle_nlp(p, u, c, "gmath", "seqfma")
    x = problem.vector_to_xdict(npz["%s/x" % name].copy(), p["M"], p["N"], p["num_sections"])
    f, _ = O.objfunc(x)
    s, _ = O.sens(x)
    _check_against_npz(npz, name, f, s, exact=True)


def test_initial_guess_matches_golden():
    npz = np.load(GOLD_REF)
    p, u, c, x0 = helpers.example_problem()
    assert np.array_equal(problem.xdict_to_vector(x0), npz["x0/x"])


def test_example_dimensions():
    """SURVEY.md A.6: 12 sections, 66 nodes, 1003 variables, 996 constraint rows."""
    p, u, c, x0 = helpers.example_problem()
    assert (p["num_sections"], p["N"], p["M"]) == (12, 66, 78)
    O = helpers.oracle_nlp(p, u, c, "libm", "numpy")
    f, _ = O.objfunc(helpers.copy_x(x0))
    assert sum(v.size for k, v in helpers.flatten_funcs(f).items() if k != "obj") == 996
    assert sum(v.size for v in x0.values()) == 1003


def test_libm_and_gmath_flavours_agree():
    """The two flavours differ only by last-bit rounding of elementary functions."""
    p, u, c, x0 = helpers.example_problem()
    fa, _ = helpers.oracle_nlp(p, u, c, "libm", "numpy").objfunc(helpers.copy_x(x0))
    fb, _ = helpers.oracle_nlp(p, u, c, "gmath", "seqfma").objfunc(helpers.copy_x(x0))
    for k, v in helpers.flatten_funcs(fa).items():
        # angle-of-attack rows go through acos near 1 (alpha ~ 1e-5 rad): ill-conditioned by 1/sin(alpha)
        atol = 1e-11 if "alpha" in k else 5e-14
        np.testing.assert_allclose(v, helpers.flatten_funcs(fb)[k], rtol=0, atol=atol, err_msg=k)


# ---------------------------------------------------------------------------
# live against the reference's Python layer (this container only)
# ---------------------------------------------------------------------------
needs_ref = pytest.mark.skipif(not refharness.available(), reason="/root/reference not present on this machine")


@needs_ref
def test_problem_setup_matches_reference():
    """gelato_b200.problem reproduces the reference's set-up block bit for bit."""
    L = leaves.get("libm")
    pr, ur, cr = refharness.reference_setup(L)
    p, u, c, _ = helpers.example_problem()
    assert ur == u
    for k in ("mass", "position", "velocity", "quaternion", "u"):
        assert np.array_equal(np.asarray(cr["init"][k]), np.asarray(c["init"][k])), k
    assert np.array_equal(np.asarray(pr["wind_table"]), p["wind_table"])
    assert np.array_equal(np.asarray(pr["ca_table"]), p["ca_table"])
    for a, b in zip(pr["params"], p["params"]):
        for key in ("name", "time", "thrust", "massflow", "reference_area", "nozzle_area", "attitude", "engineOn",
                    "mass_jettison", "num_nodes", "timeFinishAt"):
            assert a[key] == b[key], (a["name"], key)
        assert (a["time_ref"] == b["time_ref"]) or (a["time_ref"] != a["time_ref"] and b["time_ref"] != b["time_ref"])


# every variant the GPU tier is checked on against the oracle (tests/test_gpu_parity.py), plus the
# benchmark workload itself (the example refined x15 into sections of <= 20 nodes: N = 990)
LIVE_CASES = [(v, f, 12) for v in ("example", "fuel_inclination", "all_aero", "waypoints") for f in (1, 2)]
LIVE_CASES += [("neg_area", 1, 12), ("three_stage", 1, 12), ("three_stage", 2, 12), ("iip_orbital", 1, 12),
               ("bare", 1, 12), ("example", 15, 20), ("waypoints", 3, 12)]


@needs_ref
@pytest.mark.parametrize("variant,factor,max_nodes", LIVE_CASES)
def test_oracle_matches_reference_python_layer(variant, factor, max_nodes):
    """oracle/nlp.py == /root/reference/lib/con_*.py + objfunc/sens, bit for bit,
    including the residue the in-place finite differences leave in xdict."""
    L = leaves.get("libm")
    inp = helpers.variant_inputs(variant)
    p, u, c, x0 = problem.problem_from_inputs(inp, factor=factor, max_nodes=max_nodes)
    objfunc, sens = refharness.reference_callbacks(L, p, u, c)
    O = helpers.oracle_nlp(p, u, c, "libm", "numpy")
    for x in (x0, helpers.perturbed(x0)):
        xa, xb = helpers.copy_x(x), helpers.copy_x(x)
        fa, _ = objfunc(xa)
        fb, _ = O.objfunc(xb)
        helpers.assert_funcs_equal(fa, fb)
        sa, _ = sens(xa, fa)
        sb, _ = O.sens(xb)
        helpers.assert_sens_equal(sa, sb)
        for k in xa:
            assert np.array_equal(xa[k], xb[k]), "residue left in xdict[%s] differs" % k
