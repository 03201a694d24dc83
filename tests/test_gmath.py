"""gmath.h (the deterministic FP64 elementary functions shared by the CUDA
kernels and the gmath flavour of the oracle) against mpmath at 50 digits.
Accuracy target: within 2 ulp (the reference's glibc is < 1 ulp; the parity
budget of DESIGN.md H1 is written for <= 2 ulp)."""
import ctypes
import os
import subprocess

import mpmath
import numpy as np
import pytest

import gmath_corpus

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "_build", "libgmath_shim.so")
_pd = ctypes.POINTER(ctypes.c_double)


@pytest.fixture(scope="module")
def shim():
    src = os.path.join(HERE, "gmath_host_shim.c")
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-mfma", "-shared", "-fPIC", "-o", LIB, src, "-lm"])
    return ctypes.CDLL(LIB)


def _ulps(got, want_mp):
    out = []
    for g, w in zip(got, want_mp):
        wf = float(w)
        ulp = np.spacing(abs(wf)) if wf != 0 else 5e-324
        out.append(abs(mpmath.mpf(float(g)) - w) / mpmath.mpf(float(ulp)))
    return float(max(out))


def _call1(L, name, x):
    y = np.empty_like(x)
    getattr(L, name)(x.ctypes.data_as(_pd), y.ctypes.data_as(_pd), x.size)
    return y


def _call2(L, name, a, b):
    y = np.empty_like(a)
    getattr(L, name)(a.ctypes.data_as(_pd), b.ctypes.data_as(_pd), y.ctypes.data_as(_pd), a.size)
    return y


CASES1 = [
    ("gmt_sin", mpmath.sin, (-7.0, 7.0)), ("gmt_cos", mpmath.cos, (-7.0, 7.0)), ("gmt_sin", mpmath.sin, (-1e-3, 1e-3)),
    ("gmt_cos", mpmath.cos, (-0.05, 0.05)), ("gmt_tan", mpmath.tan, (-1.5, 1.5)), ("gmt_atan", mpmath.atan, (-50.0, 50.0)),
    ("gmt_asin", mpmath.asin, (-1.0, 1.0)), ("gmt_acos", mpmath.acos, (-1.0, 1.0)), ("gmt_exp", mpmath.exp, (-30.0, 5.0)),
    ("gmt_log", mpmath.log, (1e-6, 1e6)),
]


@pytest.mark.parametrize("name,ref,rng_", CASES1)
def test_unary_accuracy(shim, name, ref, rng_):
    mpmath.mp.dps = 50
    rng = np.random.default_rng(abs(hash(name)) % 2**32)
    x = rng.uniform(rng_[0], rng_[1], 1500)
    y = _call1(shim, name, x)
    assert _ulps(y, [ref(mpmath.mpf(float(v))) for v in x]) <= 2.0


def test_atan2_and_pow_accuracy(shim):
    mpmath.mp.dps = 50
    rng = np.random.default_rng(11)
    a, b = rng.uniform(-7e6, 7e6, 1500), rng.uniform(-7e6, 7e6, 1500)
    y = _call2(shim, "gmt_atan2", a, b)
    assert _ulps(y, [mpmath.atan2(mpmath.mpf(float(p)), mpmath.mpf(float(q))) for p, q in zip(a, b)]) <= 2.0
    # the US-76 pressure law: base in (0.7, 1.3), exponent up to +-35 (Air.cpp:92-96)
    base, ex = rng.uniform(0.7, 1.3, 1500), rng.uniform(-35.0, 35.0, 1500)
    y = _call2(shim, "gmt_pow", base, ex)
    assert _ulps(y, [mpmath.power(mpmath.mpf(float(p)), mpmath.mpf(float(q))) for p, q in zip(base, ex)]) <= 2.0


def test_special_values(shim):
    x = np.array([0.0, -0.0, 1.0, -1.0])
    assert np.array_equal(_call1(shim, "gmt_sin", x[:2]), x[:2])
    assert _call1(shim, "gmt_cos", x[:1])[0] == 1.0
    assert _call1(shim, "gmt_acos", x[2:3])[0] == 0.0
    assert abs(_call1(shim, "gmt_acos", x[3:4])[0] - np.pi) < 1e-15
    assert _call2(shim, "gmt_atan2", np.array([0.0]), np.array([1.0]))[0] == 0.0
    assert abs(_call2(shim, "gmt_atan2", np.array([1.0]), np.array([0.0]))[0] - np.pi / 2) < 1e-15
    assert _call1(shim, "gmt_exp", x[:1])[0] == 1.0


def test_fast_paths_equal_the_complete_functions(shim):
    """gm_atan2 / gm_pow send the common case (normal operands, moderate exponents) straight to the range reduction
    and everything else to gm_atan2_slow / gm_pow_slow, which are the complete functions.  Both routes must give the
    same bits: random operands over the whole exponent range, every pairing of the special values, and operands
    around the dispatch thresholds."""
    rng = np.random.default_rng(5)
    special = np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, np.nan, 5e-324, -5e-324, 2.2250738585072014e-308,
                        1.7976931348623157e308, -1.7976931348623157e308, 2.0 ** -27, 2.0 ** 26, 2.0 ** 25, 2.0 ** -26,
                        2.0 ** 66, 0.5, 2.0, 3.0, -3.0, 1.0 + 2.0 ** -52, 1.0 - 2.0 ** -53])
    a = np.concatenate((np.repeat(special, special.size), rng.standard_normal(200000) * 10.0 ** rng.uniform(-320, 308, 200000),
                        rng.standard_normal(200000) * 2.0 ** rng.integers(-30, 30, 200000)))
    b = np.concatenate((np.tile(special, special.size), rng.standard_normal(200000) * 10.0 ** rng.uniform(-320, 308, 200000),
                        rng.standard_normal(200000) * 2.0 ** rng.integers(-30, 30, 200000)))
    with np.errstate(all="ignore"):
        for fast, slow in (("gmt_atan2", "gmt_atan2_slow"), ("gmt_pow", "gmt_pow_slow")):
            x, y = _call2(shim, fast, a, b), _call2(shim, slow, a, b)
            same = (x.view(np.uint64) == y.view(np.uint64)) | (np.isnan(x) & np.isnan(y))
            assert same.all(), (fast, a[~same][:5], b[~same][:5], x[~same][:5], y[~same][:5])
        # pow with the operands the atmosphere uses (base around 1, exponents -35 .. 35)
        base, ex = rng.uniform(0.2, 1.6, 200000), rng.uniform(-35.0, 35.0, 200000)
        x, y = _call2(shim, "gmt_pow", base, ex), _call2(shim, "gmt_pow_slow", base, ex)
        assert np.array_equal(x.view(np.uint64), y.view(np.uint64))


def test_shared_reciprocal_division_is_the_ieee_quotient(shim):
    """gm_div_by(a, gm_rcp(d)) -- one reciprocal shared by several quotients, Markstein's correction -- must give the
    bits of a / d: random operands over the whole exponent range (the guard sends the extreme ones to the plain
    division), operands with significands next to 1 and next to 2, few-bit significands, the edges of the guard's
    exponent window, zeros, infinities and NaN (tests/gmath_corpus.py: division_operands)."""
    a, d = gmath_corpus.division_operands(np.random.default_rng(9), 2_000_000)
    with np.errstate(all="ignore"):
        got, want = _call2(shim, "gmt_div_by", a, d), a / d
    same = (got.view(np.uint64) == want.view(np.uint64)) | (np.isnan(got) & np.isnan(want))
    assert same.all(), (a[~same][:5], d[~same][:5], got[~same][:5], want[~same][:5])
