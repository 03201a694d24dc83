"""gmath.h over the whole double range, on the host and on the device.

DESIGN.md H1 rests on gmath.h giving the same bits on the host (g++) and on the device (nvcc): the oracle's gmath
flavour, the host emulator and the golden fixtures are host builds, and the kernels are trusted because they agree
with them.  The device runs code the host never runs (coefficients from __constant__ memory, __drcp_rn, __dsqrt_rn,
__fma_rn, the __noinline__ call forms, its own integer conversions), so the check is direct: every entry point of
tests/gmath_shim.h, built once with gcc (tests/gmath_host_shim.c) and once with the library's nvcc flags
(tests/gmath_device_shim.cu), on the corpus of tests/gmath_corpus.py (~10^6 inputs per entry point).

CPU and GPU: each function against mpmath on a fixed subsample of the corpus (<= 2 ulp, DESIGN.md H1), the special
values against the C99 results glibc gives, and invariants on the whole corpus.  End to end: the Earth-rotation
leaves at t up to 1e25 s against glibc."""
import ctypes
import math
import os
import re
import subprocess

import mpmath
import numpy as np
import pytest

import gmath_corpus as C

HERE = os.path.dirname(os.path.abspath(__file__))
BUILD = os.path.join(HERE, "_build")
_pd = ctypes.POINTER(ctypes.c_double)

# (shape, name) of every entry point, in the order of GMATH_SHIM_ENTRIES
ENTRIES = re.findall(r"^\s*(U2|U|B|T)\((\w+),", open(os.path.join(HERE, "gmath_shim.h")).read(), re.M)
N_IN = {"U": 1, "U2": 1, "B": 2, "T": 3}
N_OUT = {"U": 1, "U2": 2, "B": 1, "T": 1}
ULP_BOUND = 2.0
N_SAMPLE = 20_000


@pytest.fixture(scope="module")
def host():
    lib = os.path.join(BUILD, "libgmath_shim.so")
    os.makedirs(BUILD, exist_ok=True)
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-mfma", "-shared", "-fPIC", "-o", lib,
                           os.path.join(HERE, "gmath_host_shim.c"), "-lm"])
    return ctypes.CDLL(lib)


@pytest.fixture(scope="module")
def device_lib():
    """The device shim, built with the library's own nvcc flags (this needs nvcc, not a GPU)."""
    from gelato_b200 import engine

    lib = os.path.join(BUILD, "libgmath_device_shim.so")
    os.makedirs(BUILD, exist_ok=True)
    subprocess.check_call(["nvcc"] + engine.NVCC_FLAGS + ["-o", lib, os.path.join(HERE, "gmath_device_shim.cu")])
    return lib


def inputs(shape, name):
    if N_IN[shape] == 1:
        return (C.unary(name),)
    if N_IN[shape] == 2:
        return C.binary(name)
    return C.ternary(name)


def run(lib, shape, name, args, device=False):
    """Outputs of entry point gmt_<name> of `lib` on the input arrays `args`."""
    args = [np.ascontiguousarray(a, dtype=np.float64) for a in args]
    outs = [np.empty_like(args[0]) for _ in range(N_OUT[shape])]
    fn = getattr(lib, "gmt_" + name)
    fn.restype = ctypes.c_int if device else None
    err = fn(*[a.ctypes.data_as(_pd) for a in args + outs], ctypes.c_int(args[0].size))
    if device:
        assert err == 0, "gmt_%s: CUDA error %d" % (name, err)
    return outs


def same_bits(x, y):
    """Equal bits, or NaN on both sides (the payload is ignored); signed zeros must match."""
    return (x.view(np.uint64) == y.view(np.uint64)) | (np.isnan(x) & np.isnan(y))


def hexs(v):
    return [float(t).hex() for t in np.atleast_1d(v)]


# ---- the reference ----------------------------------------------------------------------------------------------

# The precision of every mpmath reference (mpmath.workdps(DPS) around each use; mpmath reduces large trigonometric
# arguments exactly at any precision, so 40 digits hold up to 1.8e308)
DPS = 40
with mpmath.workdps(DPS):
    _OVERFLOW = mpmath.ldexp(mpmath.mpf(2) - mpmath.ldexp(1, -53), 1023)  # |result| from which the double is inf


def ulp_error(got, want):
    """|got - want| in ulps of the true result `want` (an mpf, or +-inf where it lies beyond the double range); where
    it is subnormal, in ulps of the smallest subnormal."""
    if mpmath.isinf(want) or abs(want) >= _OVERFLOW:
        return 0.0 if got == (math.inf if want > 0 else -math.inf) else math.inf
    if not math.isfinite(got):
        return math.inf
    if want == 0:
        return 0.0 if got == 0 else float(abs(mpmath.mpf(got)) / mpmath.ldexp(1, -1074))
    e = mpmath.frexp(want)[1]  # |want| in [2^(e-1), 2^e)
    return float(abs(mpmath.mpf(got) - want) / mpmath.ldexp(1, max(e - 53, -1074)))


def _exp_ref(x):
    if x > 710:
        return mpmath.inf
    if x < -746:
        return mpmath.mpf(0)
    return mpmath.exp(x)


def _pow_ref(x, y):
    ax = abs(x)
    with mpmath.workprec(64):
        z = y * mpmath.log(ax, 2)
    if z > 1025:
        mag = mpmath.inf
    elif z < -1080:
        mag = mpmath.mpf(0)
    else:
        mag = mpmath.power(ax, y)
    return -mag if (x < 0 and int(y) % 2) else mag


# name -> (reference of the mpf arguments, domain mask of the float inputs)
def _fin(*a):
    m = np.ones(a[0].shape, bool)
    for v in a:
        m &= np.isfinite(v)
    return m


REFS = {
    "sin": (mpmath.sin, lambda a: _fin(a)),
    "cos": (mpmath.cos, lambda a: _fin(a)),
    "tan": (mpmath.tan, lambda a: _fin(a)),
    "atan": (mpmath.atan, lambda a: _fin(a)),
    "asin": (mpmath.asin, lambda a: np.abs(a) <= 1.0),
    "acos": (mpmath.acos, lambda a: np.abs(a) <= 1.0),
    "exp": (_exp_ref, lambda a: _fin(a)),
    "log": (mpmath.log, lambda a: _fin(a) & (a > 0)),
    "atan2": (mpmath.atan2, lambda a, b: _fin(a, b) & (a != 0) & (b != 0)),
    # a positive base, or a negative one with an integer exponent; the result inside or beyond the double range
    "pow": (_pow_ref, lambda a, b: _fin(a, b) & (a != 0) & (b != 0) & ((a > 0) | (np.floor(b) == b)) & (a != 1)),
    # the documented precondition |xl| << |x|: exp of the exact sum
    "exp_dd": (lambda x, xl: _exp_ref(x + xl), lambda a, b: _fin(a, b) & (np.abs(b) <= np.abs(a) * 2.0 ** -40)),
}


def subsample(name, args, mask):
    """A fixed subsample of about N_SAMPLE inputs in the function's domain: the trigonometric functions take all the
    reduction's worst case and a quarter from the doubles nearest k pi/2, the rest comes from the whole corpus."""
    rng = np.random.default_rng(7)
    idx = np.flatnonzero(mask)
    pick = rng.choice(idx, min(idx.size, N_SAMPLE), replace=False)
    out = [a[pick] for a in args]
    if name in ("sin", "cos", "tan"):
        hard = C.pio2_multiples()
        hard = np.concatenate((rng.choice(hard, N_SAMPLE // 4, replace=False), C.around([C.REDUCTION_WORST], 4)))
        out = [np.concatenate((out[0], hard))]
    return out


def max_ulp(host, name):
    """(largest error in ulps, its inputs, the value) of gmt_<name> over its subsample."""
    ref, dom = REFS[name]
    shape = "B" if name in ("atan2", "pow", "exp_dd") else "U"
    args = inputs(shape, name)
    sub = subsample(name, args, dom(*args))
    got = run(host, shape, name, sub)[0]
    worst = (0.0, None, None)
    with mpmath.workdps(DPS):
        for i in range(got.size):
            e = ulp_error(float(got[i]), ref(*[mpmath.mpf(float(a[i])) for a in sub]))
            if e > worst[0]:
                worst = (e, [float(a[i]) for a in sub], float(got[i]))
    return worst


@pytest.mark.parametrize("name", sorted(REFS))
def test_accuracy_over_the_whole_domain(host, name):
    """<= 2 ulp against mpmath on the whole finite domain (the reduction of arguments up to 1e308 included)."""
    err, args, got = max_ulp(host, name)
    assert err <= ULP_BOUND, (name, err, hexs(args), float(got).hex())


def test_log_dd_is_a_double_double_logarithm(host):
    """gm_log_dd (the logarithm under pow): hi within 2 ulp, hi + lo within 2^-58 relative of log x (measured:
    2^-59.5) -- the six bits beyond hi that keep pow within 2 ulp for |y log x| up to 745."""
    x = C.unary("log_dd")
    rng = np.random.default_rng(3)
    x = rng.choice(x[np.isfinite(x) & (x > 0) & (x != 1.0)], 5000, replace=False)
    hi, lo = run(host, "U2", "log_dd", (x,))
    worst_hi = worst_dd = 0.0
    with mpmath.workdps(DPS):
        for v, h, l in zip(x, hi, lo):
            w = mpmath.log(mpmath.mpf(float(v)))
            worst_hi = max(worst_hi, ulp_error(float(h), w))
            worst_dd = max(worst_dd, float(abs(mpmath.mpf(float(h)) + mpmath.mpf(float(l)) - w) / abs(w)))
    assert worst_hi <= ULP_BOUND and worst_dd <= 2.0 ** -58, (worst_hi, worst_dd)


def test_primitives_are_the_ieee_operations(host):
    """gm_sqrt and gm_div_by(a, gm_rcp(d)) give the bits of the IEEE square root and quotient."""
    with np.errstate(all="ignore"):
        x = C.unary("sqrt")
        assert same_bits(run(host, "U", "sqrt", (x,))[0], np.sqrt(x)).all()
        a, d = C.binary("div_by")
        got, want = run(host, "B", "div_by", (a, d))[0], a / d
    same = same_bits(got, want)
    assert same.all(), (hexs(a[~same][:5]), hexs(d[~same][:5]), hexs(got[~same][:5]), hexs(want[~same][:5]))


def test_forms_of_a_function_give_the_same_bits(host):
    """The call forms, the _inl forms, sincos and the slow routes of atan2 / pow are the same function."""
    x = C.unary("sin")
    s, c = run(host, "U2", "sincos", (x,))
    for shape, name, want in (("U", "sin", s), ("U", "sin_inl", s), ("U", "cos", c), ("U", "cos_inl", c)):
        got = run(host, shape, name, (C.unary("sin"),))[0]
        assert same_bits(got, want).all(), name
    si, ci = run(host, "U2", "sincos_inl", (x,))
    assert same_bits(si, s).all() and same_bits(ci, c).all()
    # gm_sincos_small_inl, the hot path's form for atan2 results: the same bits below 2^50, NaN from there on
    small = np.abs(x) < C.REM_PIO2_LARGE
    ss, cs = run(host, "U2", "sincos_small_inl", (x,))
    assert same_bits(ss[small], s[small]).all() and same_bits(cs[small], c[small]).all()
    assert np.isnan(ss[~small]).all() and np.isnan(cs[~small]).all()
    x = C.unary("exp")
    assert same_bits(run(host, "U", "exp_inl", (x,))[0], run(host, "U", "exp", (x,))[0]).all()
    with np.errstate(all="ignore"):
        for fn in ("atan2", "pow"):
            a, b = C.binary(fn)
            want = run(host, "B", fn, (a, b))[0]
            for form in ("_inl", "_slow"):
                assert same_bits(run(host, "B", fn + form, (a, b))[0], want).all(), fn + form


def _kind(v):
    """NaN / +-inf / +-0 / finite of either sign: what a special value must match."""
    v = np.asarray(v, dtype=np.float64)
    k = np.where(v > 0, 1, np.where(v < 0, 2, 3))
    k = np.where(v == 0, np.where(np.signbit(v), 4, 5), k)
    k = np.where(np.isinf(v), np.where(v > 0, 6, 7), k)
    return np.where(np.isnan(v), 8, k)


def test_special_values(host):
    """On the special values (+-0, +-inf, NaN, the smallest subnormal and normal, the largest double, +-1, +-0.5, +-2;
    every pair for atan2 and pow) each function gives what C99 Annex F prescribes (checked against glibc through
    numpy): NaN, the infinities and the signed zeros exactly, and the exact results (cos 0, exp 0, log 1, pow's
    special cases) bit for bit."""
    s = C.SPECIAL
    with np.errstate(all="ignore"):
        for name, want in (("sin", np.sin(s)), ("cos", np.cos(s)), ("tan", np.tan(s)), ("atan", np.arctan(s)),
                           ("asin", np.arcsin(s)), ("acos", np.arccos(s)), ("exp", np.exp(s)), ("log", np.log(s))):
            got = run(host, "U", name, (s,))[0]
            assert (_kind(got) == _kind(want)).all(), (name, hexs(s), hexs(got), hexs(want))
            exact = (want == 0) | np.isinf(want) | (np.abs(want) == 1.0)
            assert same_bits(got[exact], want[exact]).all(), (name, hexs(s[exact]), hexs(got[exact]))
        a, b = np.repeat(s, s.size), np.tile(s, s.size)
        for name, want in (("atan2", np.arctan2(a, b)), ("pow", np.power(a, b))):
            got = run(host, "B", name, (a, b))[0]
            bad = _kind(got) != _kind(want)
            assert not bad.any(), (name, hexs(a[bad]), hexs(b[bad]), hexs(got[bad]), hexs(want[bad]))
            exact = (want == 0) | np.isinf(want) | (want == 1.0) | ((a == 0) | np.isinf(a) | np.isinf(b)) & ~np.isnan(want)
            exact &= (name == "pow") | (want == 0)
            ok = same_bits(got[exact], want[exact])
            assert ok.all(), (name, hexs(a[exact][~ok]), hexs(b[exact][~ok]), hexs(got[exact][~ok]))
        acos = run(host, "U", "acos", (np.array([1.0, -1.0, 0.0]),))[0]
        assert acos[0] == 0.0 and not np.signbit(acos[0]) and acos[1] == np.pi and acos[2] == np.pi / 2


def test_invariants_on_the_whole_corpus(host):
    """|sin| <= 1 and |cos| <= 1 everywhere; a finite input whose true result lies inside the double range never
    gives inf or NaN."""
    x = C.unary("sin")
    s, c = run(host, "U2", "sincos", (x,))
    fin = np.isfinite(x)
    assert (np.abs(s[fin]) <= 1.0).all() and (np.abs(c[fin]) <= 1.0).all()
    with np.errstate(all="ignore"):
        checks = [("U", "sin", None), ("U", "cos", None), ("U", "tan", None), ("U", "atan", None),
                  ("U", "asin", lambda a: np.abs(a) <= 1.0), ("U", "acos", lambda a: np.abs(a) <= 1.0),
                  ("U", "exp", lambda a: a <= 709.782712893384), ("U", "log", lambda a: a > 0),
                  ("U", "sqrt", lambda a: a >= 0), ("B", "atan2", None),
                  ("B", "pow", lambda a, b: (a > 0) & (np.abs(b * np.log2(np.abs(a))) < 1020.0)),
                  ("B", "exp_dd", lambda a, b: (a <= 709.0) & (np.abs(b) <= np.abs(a) * 2.0 ** -40)),
                  ("B", "div_by", lambda a, b: (b != 0) & (np.abs(a / b) < 1e308))]
        for shape, name, dom in checks:
            args = inputs(shape, name)
            m = _fin(*args)
            if dom is not None:
                m &= dom(*args)
            got = run(host, shape, name, args)[0]
            bad = m & ~np.isfinite(got)
            assert not bad.any(), (name, [hexs(a[bad][:5]) for a in args], hexs(got[bad][:5]))


def test_device_shim_builds(device_lib):
    """The device shim compiles with the library's flags and exports every entry point."""
    syms = subprocess.check_output(["nm", "-D", "--defined-only", device_lib], text=True)
    assert sorted(re.findall(r" T gmt_(\w+)$", syms, re.M)) == sorted(name for _, name in ENTRIES)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,name", ENTRIES, ids=[name for _, name in ENTRIES])
def test_device_equals_host(host, device_lib, shape, name):
    """Every entry point gives the same bits on the device as on the host on its whole corpus."""
    dev = ctypes.CDLL(device_lib)
    args = inputs(shape, name)
    with np.errstate(all="ignore"):
        want = run(host, shape, name, args)
    got = run(dev, shape, name, args, device=True)
    for k, (g, w) in enumerate(zip(got, want)):
        same = same_bits(g, w)
        bad = np.flatnonzero(~same)[:8]
        assert same.all(), ("gmt_%s output %d: %d of %d differ" % (name, k, (~same).sum(), same.size),
                            [(hexs([a[i] for a in args]), float(g[i]).hex(), float(w[i]).hex()) for i in bad])


# ---- end to end: the Earth-rotation leaves at large t -----------------------------------------------------------

T_LARGE = 10.0 ** np.arange(6.0, 26.0)
POS = np.array([6378137.0 * 0.6, -6378137.0 * 0.7, 6378137.0 * 0.39])


def _assert_like_glibc(got, want):
    """Within 4 ulp of |r| of the glibc flavour."""
    tol = 4 * np.spacing(np.linalg.norm(POS))
    err = np.abs(np.asarray(got) - np.asarray(want)).max(axis=-1)
    assert (err <= tol).all(), (T_LARGE[err > tol], err[err > tol])


def test_coordinate_leaves_at_large_t_oracle():
    """The oracle's gmath flavour of eci2ecef / ecef2eci against its glibc flavour at t = 1e6 .. 1e25 s (omega t up
    to 7e20 goes through the argument reduction)."""
    from oracle import leaves

    g, m = leaves.get("gmath").coordinate_c, leaves.get("libm").coordinate_c
    for fn in ("eci2ecef", "ecef2eci"):
        got = np.array([getattr(g, fn)(POS, t) for t in T_LARGE])
        want = np.array([getattr(m, fn)(POS, t) for t in T_LARGE])
        _assert_like_glibc(got, want)


@pytest.mark.gpu
def test_coordinate_leaves_at_large_t_device():
    """The drop-in lib.coordinate_c.eci2ecef / ecef2eci on the device against the glibc flavour, t = 1e6 .. 1e25 s."""
    from gelato_b200.lib import coordinate_c
    from oracle import leaves

    m = leaves.get("libm").coordinate_c
    pos = np.broadcast_to(POS, (T_LARGE.size, 3))
    for fn in ("eci2ecef", "ecef2eci"):
        got = getattr(coordinate_c, fn)(pos, T_LARGE)
        want = np.array([getattr(m, fn)(POS, t) for t in T_LARGE])
        _assert_like_glibc(got, want)


@pytest.mark.gpu
def test_rotation_inlined_in_a_kernel_at_large_t():
    """The large-argument branch where the NLP kernels meet it: inlined into rotq_part (omega t and omega t / 2), here
    through the dynamics_velocity leaf kernel, against the oracle's gmath flavour bit for bit, with omega t from 7e-3
    to 7e19 (across 2^50) and t within 8 ulp of where omega t or omega t / 2 reaches 2^50."""
    import helpers
    from gelato_b200.lib import dynamics_c
    from oracle import leaves

    inp = helpers.example_inputs()
    wind, ca = np.asarray(inp["wind_table"], dtype=float), np.asarray(inp["ca_table"], dtype=float)
    units = np.array([27442.0, 6378137.0, 1000.0])
    omega = 7.2921151467e-5  # physics.h: P_OMEGA; rotq_part reduces omega t and omega t / 2
    t = np.concatenate((10.0 ** np.linspace(2.0, 24.0, 300), C.around(C.REM_PIO2_LARGE / omega * np.array([1.0, 2.0]))))
    n = t.size
    rng = np.random.default_rng(12)
    pos = np.tile(POS / units[1] * 1.01, (n, 1))
    vel = rng.normal(size=(n, 3)) * 2.0
    q = rng.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    mass = rng.uniform(0.05, 1.0, n)
    a = (mass, pos, vel, q, t, np.array([420000.0, 140.9, 2.21, 0.0, 0.68]), wind, ca, units)
    got, want = np.asarray(dynamics_c.dynamics_velocity(*a)), np.asarray(leaves.get("gmath").dynamics_c.dynamics_velocity(*a))
    same = same_bits(got.ravel(), want.ravel()).reshape(got.shape).all(axis=-1)
    assert same.all(), (hexs(t[~same][:5]), got[~same][:3], want[~same][:3])
