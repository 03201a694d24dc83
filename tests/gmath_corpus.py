"""One seeded input corpus for the gmath.h entry points of tests/gmath_shim.h, shared by the host checks
(tests/test_gmath.py, tests/test_gmath_device.py against mpmath) and the device check (device == host).

Per function: ~10^6 random bit patterns over all finite doubles (both signs, subnormals included), the special values
(every pair of them for the two-argument functions), the doubles within 8 ulp of every dispatch threshold of gmath.h,
the ranges the kernels use sampled densely and, for the trigonometric functions, the hard cases of the argument
reduction."""
import functools

import mpmath
import numpy as np

N_RANDOM = 1_000_000

SPECIAL = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 5e-324, -5e-324, 2.2250738585072014e-308, -2.2250738585072014e-308,
                    1.7976931348623157e308, -1.7976931348623157e308, 1.0, -1.0, 0.5, -0.5, 2.0, -2.0])

# |x| from which gm_rem_pio2 takes the Payne-Hanek reduction (gmath.h: GM_REM_PIO2_LARGE)
REM_PIO2_LARGE = 2.0 ** 50
# the classic worst case of the reduction: its remainder is 4.687e-19
REDUCTION_WORST = float(mpmath.ldexp(6381956970095103, 797))


def around(v, k=8):
    """The doubles within k ulp of each value of v, both signs."""
    u = np.abs(np.atleast_1d(np.asarray(v, dtype=np.float64))).view(np.int64)
    bits = (u[:, None] + np.arange(-k, k + 1, dtype=np.int64)[None, :]).ravel()
    bits = bits[(bits >= 0) & (bits < 0x7ff0000000000000)]
    x = bits.view(np.float64)
    return np.concatenate((x, -x))


def random_finite(rng, n):
    """n random bit patterns over all finite doubles: both signs, subnormals included, no inf or NaN."""
    u = rng.integers(0, 1 << 63, n, dtype=np.uint64) | (rng.integers(0, 2, n, dtype=np.uint64) << np.uint64(63))
    bad = (u & np.uint64(0x7ff0000000000000)) == np.uint64(0x7ff0000000000000)
    u[bad] &= np.uint64(0x800fffffffffffff)  # the few inf / NaN patterns become subnormals
    return u.view(np.float64)


def _rng(name):
    return np.random.default_rng(sum(ord(ch) * 131 ** i for i, ch in enumerate(name)) % 2 ** 32)


@functools.lru_cache(maxsize=None)
def pio2_multiples():
    """The doubles nearest k pi/2 (and their neighbours) for k = 1 .. 1000 and 600 k log-uniform up to 2^60."""
    rng = np.random.default_rng(2)
    ks = list(range(1, 1001)) + [int(v) for v in np.unique(np.floor(2.0 ** rng.uniform(10, 60, 600)))]
    with mpmath.workprec(256):
        x = np.array([float(k * mpmath.pi / 2) for k in ks])
    return around(x, 2)


def trig_hard(rng):
    return np.concatenate((pio2_multiples(), around([REDUCTION_WORST], 4),
                           10.0 ** rng.uniform(6, 308, 100_000) * rng.choice([-1.0, 1.0], 100_000)))


def _unary_extra(name, rng):
    base = name.split("_")[0]
    if base in ("sin", "cos", "sincos", "tan"):
        dense = [rng.uniform(-7.0, 7.0, 50_000), rng.uniform(-1e-3, 1e-3, 20_000), rng.uniform(-0.05, 0.05, 20_000),
                 rng.uniform(-1.5, 1.5, 20_000)]
        thr = around([np.pi / 4, REM_PIO2_LARGE, 2.0 ** 51 * np.pi / 2, np.pi / 2, np.pi, 2.0 ** -27])
        return np.concatenate(dense + [thr, trig_hard(rng)])
    if base == "atan":
        return np.concatenate((rng.uniform(-50.0, 50.0, 50_000), around([2.0 ** -27, 0.4375, 0.6875, 1.1875, 2.4375, 2.0 ** 66])))
    if base in ("asin", "acos"):
        return np.concatenate((rng.uniform(-1.0, 1.0, 50_000), around([1.0, 0.5, 2.0 ** -27, 2.0 ** -1022], 8)))
    if base == "exp":
        # overflow guard, underflow guard, the first subnormal result (ln 2^-1022) and the last non-zero one
        return np.concatenate((rng.uniform(-30.0, 5.0, 50_000), rng.uniform(-750.0, 712.0, 50_000),
                               around([709.782712893384, 709.782712893383973096, 745.2, 708.3964185322641,
                                       745.1332191019411, 745.1332191019412])))
    if base == "log":
        sub = random_finite(rng, 50_000)
        sub = np.abs(sub.view(np.uint64) & np.uint64(0x000fffffffffffff)).view(np.float64)  # subnormals
        split = np.array([0x3ff6a09e667f3bcd], dtype=np.int64).view(np.float64)[0]  # sqrt(2)'s mantissa split
        return np.concatenate((np.exp(rng.uniform(np.log(1e-6), np.log(1e6), 50_000)), sub,
                               around(split * 2.0 ** np.arange(-1074, 1024, 37.0)), around([2.0 ** -1022, 5e-324, 1.0])))
    if base == "rcp":
        return np.concatenate((around(2.0 ** np.array([-500.0, -501.0, 500.0, 501.0])),
                               around(np.nextafter(2.0 ** np.array([-499.0, 501.0]), 0.0)), rng.uniform(-1e3, 1e3, 20_000)))
    if base == "sqrt":
        return np.concatenate((around([1.0, 2.0, 2.0 ** -1022, 5e-324, 4.0]), rng.uniform(0.0, 1e8, 20_000)))
    return np.zeros(0)


@functools.lru_cache(maxsize=None)
def unary(name):
    """The inputs of a one-argument entry point (U or U2 in tests/gmath_shim.h)."""
    rng = _rng(name)
    return np.concatenate((random_finite(rng, N_RANDOM), SPECIAL, _unary_extra(name, rng)))


def _pairs_of(v):
    return np.repeat(v, v.size), np.tile(v, v.size)


def _binary_extra(name, rng):
    base = name.split("_")[0]
    if name.startswith("atan2"):
        a, b = rng.uniform(-7e6, 7e6, 50_000), rng.uniform(-7e6, 7e6, 50_000)
        # exponent differences around +-26 (the fast path's window) and +-64 (gm_atan2_slow's cut-offs)
        n = 40_000
        x = rng.uniform(1.0, 2.0, n) * 2.0 ** rng.integers(-300, 300, n)
        k = rng.choice(np.r_[-66:-61, -28:-23, 24:29, 62:67], n).astype(np.float64)
        m = rng.choice([1.0, np.nextafter(2.0, 0.0), 1.5], n) * rng.choice([1.0, -1.0], n)
        y = m * 2.0 ** (np.floor(np.log2(x)) + k)
        x = x * rng.choice([1.0, -1.0], n)
        return np.concatenate((a, y)), np.concatenate((b, x))
    if base == "pow":
        parts = [(rng.uniform(0.7, 1.3, 50_000), rng.uniform(-35.0, 35.0, 50_000)),
                 (rng.uniform(0.2, 1.6, 50_000), rng.uniform(-35.0, 35.0, 50_000))]
        s = np.sin(rng.uniform(-np.pi, np.pi, 20_000))  # the haversine: pow(sin(.), 2)
        parts.append((s, np.full(s.size, 2.0)))
        # results inside the double range: a random base, the exponent scaled to it
        xr = np.abs(random_finite(rng, 50_000))
        xr = xr[(xr != 0.0) & (xr != 1.0)]
        yr = rng.uniform(-1.0, 1.0, xr.size) * 1070.0 / np.abs(np.log2(xr))
        parts.append((xr, yr))
        # gm_is_int around 2^51 and 2^53 with negative bases; odd and even integers, both signs of the base
        y = around([2.0 ** 51, 2.0 ** 53, 3.0, 2.0 ** 52])
        xb = np.array([-1.0, -0.5, -2.0, -1.0 - 2.0 ** -52, -1.0 + 2.0 ** -53, 1.0 + 2.0 ** -52, -0.0, 0.0, -np.inf])
        parts.append((np.repeat(xb, y.size), np.tile(y, xb.size)))
        return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])
    if name == "exp_dd":
        x = np.concatenate((rng.uniform(-745.0, 709.0, 50_000), around([709.782712893384, 745.2, 708.3964185322641])))
        return x, x * rng.uniform(-1.0, 1.0, x.size) * 2.0 ** -54
    if name == "div_by":
        return division_operands(np.random.default_rng(9), 60_000)
    return np.zeros(0), np.zeros(0)


@functools.lru_cache(maxsize=None)
def binary(name):
    """The inputs of a two-argument entry point (B in tests/gmath_shim.h)."""
    rng = _rng(name)
    a, b = random_finite(rng, N_RANDOM), random_finite(rng, N_RANDOM)
    sa, sb = _pairs_of(SPECIAL)
    ea, eb = _binary_extra(name, rng)
    return np.concatenate((a, sa, ea)), np.concatenate((b, sb, eb))


@functools.lru_cache(maxsize=None)
def ternary(name):
    """The inputs of gm_fma: random bit patterns, triples of special values, and products that cancel the addend."""
    rng = _rng(name)
    a, b, c = (random_finite(rng, N_RANDOM) for _ in range(3))
    s = SPECIAL
    sa, sb, sc = (np.repeat(s, s.size * s.size), np.tile(np.repeat(s, s.size), s.size), np.tile(s, s.size * s.size))
    x, y = rng.uniform(-2.0, 2.0, 20_000), rng.uniform(-2.0, 2.0, 20_000)
    return (np.concatenate((a, sa, x)), np.concatenate((b, sb, y)), np.concatenate((c, sc, -(x * y))))


def division_operands(rng, n):
    """Operand pairs (a, d) for gm_div_by: random operands over +-600 binades (the guard sends the extreme ones to the
    plain division), significands next to 1 and next to 2, few-bit significands, and every pair of special values."""

    def sig(kind):
        m = rng.integers(0, 1 << 52, n, dtype=np.uint64)
        if kind == 1:
            m = (np.uint64((1 << 52) - 1) - (m & np.uint64(0xff)))
        elif kind == 2:
            m = m & np.uint64(0xff)
        elif kind == 3:
            m = m & np.uint64(0xfffff00000000)
        return m

    parts_a, parts_d = [], []
    for ka in range(4):
        for kd in range(4):
            if (ka, kd) not in ((0, 0), (1, 1), (2, 2), (0, 1), (1, 0), (0, 2), (2, 0), (3, 3), (0, 3)):
                continue
            ea = rng.integers(1023 - 600, 1023 + 600, n).astype(np.uint64)
            ed = rng.integers(1023 - 600, 1023 + 600, n).astype(np.uint64)
            sa = rng.integers(0, 2, n).astype(np.uint64) << np.uint64(63)
            sd = rng.integers(0, 2, n).astype(np.uint64) << np.uint64(63)
            parts_a.append((sa | (ea << np.uint64(52)) | sig(ka)).view(np.float64))
            parts_d.append((sd | (ed << np.uint64(52)) | sig(kd)).view(np.float64))
    special = np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, np.nan, 5e-324, 2.2250738585072014e-308, 1.7976931348623157e308,
                        1e-8, 6378137.0, 1000.0, 3.0, 1.0 / 3.0])
    parts_a.append(np.repeat(special, special.size))
    parts_d.append(np.tile(special, special.size))
    # the edges of the guard's exponent window (biased exponents 523 .. 1523) on either operand
    edge = around(2.0 ** np.array([-500.0, 500.0]), 8)
    edge = np.concatenate((edge, around(np.nextafter(2.0 ** np.array([-500.0, 501.0]), 0.0), 8)))
    other = rng.uniform(1.0, 2.0, edge.size) * rng.choice([1.0, -1.0], edge.size)
    parts_a += [edge, other]
    parts_d += [other, edge]
    return np.concatenate(parts_a), np.concatenate(parts_d)
