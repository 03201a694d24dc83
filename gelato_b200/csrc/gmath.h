/* gmath.h -- deterministic binary64 elementary functions for host AND device.
 *
 * Why this exists (DESIGN.md "H1"): the reference differentiates its physics
 * with forward finite differences, dx = 1e-8
 * (/root/reference/Trajectory_Optimization.py:167), so a 1-ulp disagreement in
 * one sin()/atan2()/pow() call moves a Jacobian entry by ~1e-8 relative -- two
 * orders above the 1e-10 parity tolerance.  CUDA's libdevice and glibc's libm
 * do not agree to the last bit, so the GPU path and the gmath flavour of the
 * CPU oracle both call THESE functions.  They are built only from IEEE-754
 * correctly rounded primitives (+ - * / sqrt fma) and integer bit operations,
 * therefore g++ (-ffp-contract=off) and nvcc (-fmad=false) produce identical
 * bits.  Accuracy is <= 2 ulp for every function over the whole double range
 * (measured against mpmath in tests/test_gmath_device.py; maxima in DESIGN.md H1).
 *
 * The polynomial tables in gmath_coeffs.inc are generated from first
 * principles by tools/gen_gmath_coeffs.py (mpmath Chebyshev fits).
 *
 * Reference call sites these replace: sin/cos/atan2/sqrt in
 * /root/reference/src/Earth.cpp:49-61 and Coordinate.cpp:41-98, pow/exp/sqrt in
 * Air.cpp:71-111, acos in wrapper_utils.hpp:109 and Coordinate.cpp:208-231,
 * asin/tan/atan2 in iip.cpp:131-143.
 */
#ifndef GELATO_B200_GMATH_H_
#define GELATO_B200_GMATH_H_

#include <stdint.h>
#include <string.h>

#include "gmath_coeffs.inc"
#include "gmath_table.inc"

/* The coefficients as operands.  Host: the literals of gmath_coeffs.inc.  Device: the same literals read from one
 * table in __constant__ memory (gmath_table.inc) -- identical values, so identical results; what changes is the
 * instruction count: a 64-bit literal costs two 32-bit immediate moves per use, a constant-bank operand none
 * (ncu r02a: moves were 27 % of the instructions the Jacobian kernel executed, as many as its FP64 arithmetic). */
#if defined(__CUDACC__)
static __constant__ double gm_tab[GM_TAB_N] = GM_TAB_INIT;
static __constant__ uint64_t gm_2opi_dev[GM_2OPI_N] = GM_2OPI_INIT;
#endif
static const uint64_t gm_2opi_host[GM_2OPI_N] = GM_2OPI_INIT;
#if defined(__CUDA_ARCH__)
#define GMC(name) gm_tab[GMT_##name]
#define GM_2OPI(j) gm_2opi_dev[j]
#else
#define GMC(name) GM_##name
#define GM_2OPI(j) gm_2opi_host[j]
#endif

#if defined(__CUDACC__)
#define GM_HD static __host__ __device__ inline
/* The large elementary functions exist in two forms.  `gm_xxx` is a real call on the device (__noinline__): a
 * right-hand side evaluates ~20 of them, and with every copy inlined the Jacobian kernel was 365 KB of SASS -- far
 * beyond the SM instruction cache (ncu round 1: stall_no_instruction 8.3 per issue).  `gm_xxx_inl` is the same body
 * forced inline, for the two functions that ARE the hot path (physics.h: pos_part, rotq_part; themselves called
 * once per item): there a call costs more in argument moves and spills than the body is worth sharing (ncu r02a:
 * 18 % of the executed instructions were register moves). */
#define GM_HD_CALL static __host__ __device__ __noinline__
#define GM_HD_INL static __host__ __device__ __forceinline__
#else
#define GM_HD static inline
#define GM_HD_CALL static inline
#define GM_HD_INL static inline
#endif

/* ---- primitives ------------------------------------------------------- */
/* IEEE division.  On the device a quotient is ~30 instructions inline and the NLP kernels contain a few
 * hundred of them; as a call each exists once and the kernels' instruction footprint shrinks (measured:
 * k_jacobian 0.153 -> 0.150 ms; GM_DIV_CALLS=0 restores the inline form; profiles/r01r_div_ab.txt). */
#ifndef GM_DIV_CALLS
#define GM_DIV_CALLS 1
#endif
#if GM_DIV_CALLS
GM_HD_CALL double gm_div(double a, double b) { return a / b; }
#else
GM_HD double gm_div(double a, double b) { return a / b; }
#endif

GM_HD double gm_fma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
  return __fma_rn(a, b, c);
#else
  return __builtin_fma(a, b, c);
#endif
}

GM_HD double gm_sqrt(double x) {
#if defined(__CUDA_ARCH__)
  return __dsqrt_rn(x);
#else
  return __builtin_sqrt(x);
#endif
}

GM_HD uint64_t gm_d2u(double x) {
#if defined(__CUDA_ARCH__)
  return (uint64_t)__double_as_longlong(x);
#else
  uint64_t u;
  memcpy(&u, &x, sizeof u);
  return u;
#endif
}

GM_HD double gm_u2d(uint64_t u) {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double((long long)u);
#else
  double x;
  memcpy(&x, &u, sizeof x);
  return x;
#endif
}

/* ---- division by a shared denominator ---------------------------------------------------------------
 * Several quotients with the same denominator (a vector over its norm, an acceleration over the mass, every
 * finite-difference quotient over dx) need only ONE reciprocal: with r = RN(1/d) (IEEE reciprocal), q = RN(a r),
 * rem = a - q d (exact in one fused multiply-add) and q' = RN(q + rem r), q' is the correctly rounded a / d
 * (Markstein's theorem; holds whenever no intermediate over- or underflows).  The result is the IEEE quotient --
 * the bits `a / d` gives -- for operands in the guarded exponent range; anything else (zeros, infinities, NaN,
 * tiny or huge operands) takes the plain division.  tests/test_gmath.py checks the equality on 10^7 operand pairs,
 * adversarial significands included (6 x 10^8 more in the build container: profiles/r02_division.txt).
 * On the device a quotient costs 3 FP64 instructions + the guard instead of the ~20 of the division routine
 * (ncu r02e: division was 17 % of the instructions the Jacobian kernel executed). */
#ifndef GM_SHARED_RCP
#define GM_SHARED_RCP 1
#endif
typedef struct GmRcp {
  double d, r; /* denominator, RN(1 / d) */
  int ok;      /* d is a normal number with an exponent in [-500, 500] */
} GmRcp;
GM_HD GmRcp gm_rcp(double d) {
  GmRcp R;
  R.d = d;
#if defined(__CUDA_ARCH__)
  R.r = __drcp_rn(d);
#else
  R.r = 1.0 / d;
#endif
  R.ok = (uint32_t)((gm_d2u(d) >> 52) & 0x7ffu) - 523u < 1001u;
  return R;
}
GM_HD double gm_div_by(double a, const GmRcp R) {
#if GM_SHARED_RCP
  if (R.ok && (uint32_t)((gm_d2u(a) >> 52) & 0x7ffu) - 523u < 1001u) {
    const double q = a * R.r;
    const double rem = gm_fma(-q, R.d, a);
    return gm_fma(rem, R.r, q);
  }
#endif
  return gm_div(a, R.d);
}

#define GM_SIGN_MASK 0x8000000000000000ull
#define GM_ABS_MASK 0x7fffffffffffffffull
#define GM_INF_BITS 0x7ff0000000000000ull

/* high word of the 128-bit product; leading zeros of a non-zero word */
GM_HD uint64_t gm_umulhi(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}
GM_HD int gm_clz64(uint64_t a) {
#if defined(__CUDA_ARCH__)
  return __clzll((long long)a);
#else
  return __builtin_clzll(a);
#endif
}

GM_HD double gm_fabs(double x) { return gm_u2d(gm_d2u(x) & GM_ABS_MASK); }
GM_HD double gm_copysign(double mag, double sgn) {
  return gm_u2d((gm_d2u(mag) & GM_ABS_MASK) | (gm_d2u(sgn) & GM_SIGN_MASK));
}
GM_HD int gm_isnan(double x) { return (gm_d2u(x) & GM_ABS_MASK) > GM_INF_BITS; }
GM_HD double gm_nan(void) { return gm_u2d(0x7ff8000000000000ull); }
GM_HD double gm_inf(void) { return gm_u2d(GM_INF_BITS); }

/* round to nearest integer (ties to even), |x| < 2^51 */
GM_HD double gm_rint(double x) {
  const double magic = 6755399441055744.0; /* 1.5 * 2^52 */
  double t = x + magic;
  return t - magic;
}

/* ---- sin / cos / tan -------------------------------------------------- */

/* |x| from which gm_rem_pio2 takes the Payne-Hanek reduction: 2^50.  Below it k = rint(x 2/pi) < 2^50 and the
 * three pieces of pi/2 are accurate enough: measured against mpmath on [2^49, 2^50), the doubles nearest k pi/2
 * included, sin 0.76, cos 0.72, tan 1.96 ulp.  Above it they are not (the same measurement on [2^50, 2^51): sin 16.7,
 * tan 18.2 ulp), and from 2^51 pi/2 on the rint trick no longer rounds k to an integer. */
#define GM_REM_PIO2_LARGE 0x4310000000000000ull

/* x - k*pi/2 for |x| >= GM_REM_PIO2_LARGE (Payne-Hanek; correct for every finite x).  With x = m 2^E (m the 53-bit
 * significand) the bits of 2/pi before b(E-1) contribute multiples of 4 to x 2/pi, so only the 192 bits from b(E-1)
 * on are needed: m times that window, modulo 2^192, is x 2/pi modulo 4 as a fixed-point number with 190 fractional
 * bits.  The bits of 2/pi after the window add less than 2^-137 to it; the fraction of a double is never smaller
 * than 2^-62 (the worst case, 6381956970095103 2^797), so hi + lo -- the 53 + 53 bits taken from it -- is the
 * fraction to a relative 2^-75, far below an ulp of the result.
 * Integer arithmetic only up to the final product with pi/2, so host and device agree.  Returned by value, so that no
 * local of the caller has to live in memory. */
typedef struct GmRem {
  double r, rl; /* x - k pi/2 as a double-double */
  int q;        /* k mod 4 */
} GmRem;
GM_HD GmRem gm_rem_pio2_large(double x) {
  const uint64_t ux = gm_d2u(x);
  const uint64_t m = (ux & 0x000fffffffffffffull) | 0x0010000000000000ull;
  const int g = (int)((ux >> 52) & 0x7ffu) - 1075 - 2 + 64; /* bit b(E-1) in the table, whose word 0 is zeros */
  const int j = g >> 6, sh = g & 63;
  uint64_t w0 = GM_2OPI(j), w1 = GM_2OPI(j + 1), w2 = GM_2OPI(j + 2);
  if (sh) {
    w0 = (w0 << sh) | (w1 >> (64 - sh));
    w1 = (w1 << sh) | (w2 >> (64 - sh));
    w2 = (w2 << sh) | (GM_2OPI(j + 3) >> (64 - sh));
  }
  /* (a0, a1, a2) = m (w0, w1, w2) mod 2^192 */
  const uint64_t a2 = m * w2;
  const uint64_t p1 = m * w1, c2 = gm_umulhi(m, w2);
  uint64_t a1 = p1 + c2;
  uint64_t a0 = m * w0 + gm_umulhi(m, w1) + (uint64_t)(a1 < p1);
  int q = (int)(a0 >> 62);
  a0 &= 0x3fffffffffffffffull;
  uint64_t b2 = a2, b1 = a1;
  int neg = 0;
  if (a0 >> 61) { /* fraction >= 1/2: x 2/pi = (q + 1) - (1 - fraction) */
    q += 1;
    neg = 1;
    b2 = ~a2 + 1;
    b1 = ~a1 + (uint64_t)(b2 == 0);
    a0 = (~a0 + (uint64_t)(b2 == 0 && b1 == 0)) & 0x3fffffffffffffffull;
  }
  /* normalise (a0, b1, b2) so that bit 191 is set; s = the shift */
  int s = 0;
  if (a0 == 0) {
    a0 = b1;
    b1 = b2;
    b2 = 0;
    s += 64;
    if (a0 == 0) {
      a0 = b1;
      b1 = 0;
      s += 64;
    }
  }
  double hi = 0.0, lo = 0.0;
  if (a0 != 0) {
    const int z = gm_clz64(a0);
    if (z) {
      a0 = (a0 << z) | (b1 >> (64 - z));
      b1 = (b1 << z) | (b2 >> (64 - z));
    }
    s += z;
    /* fraction = hi + lo: the top 53 bits and the next 53, both exact doubles; s <= 190 keeps the scales normal */
    hi = (double)(a0 >> 11) * gm_u2d((uint64_t)(1023 - 51 - s) << 52);
    lo = (double)(((a0 & 0x7ffu) << 42) | (b1 >> 22)) * gm_u2d((uint64_t)(1023 - 104 - s) << 52);
  }
  /* (hi + lo) pi/2 in double-double */
  const double ph = hi * GMC(PIO2_1);
  const double tail = gm_fma(hi, GMC(PIO2_1), -ph) + gm_fma(hi, GMC(PIO2_2), lo * GMC(PIO2_1));
  double r0 = ph + tail;
  double r1 = (ph - r0) + tail;
  if (neg) {
    r0 = -r0;
    r1 = -r1;
  }
  if (ux & GM_SIGN_MASK) {
    r0 = -r0;
    r1 = -r1;
    q = -q;
  }
  GmRem R;
  R.r = r0;
  R.rl = r1;
  R.q = q & 3;
  return R;
}

/* x - k*pi/2 as a double-double (r, rl) for |x| < GM_REM_PIO2_LARGE: k = rint(x 2/pi) and three 53-bit pieces of
 * pi/2 (159 bits); returns k mod 4. */
GM_HD int gm_rem_pio2_small(double x, double* r, double* rl) {
  double kd = gm_rint(x * GMC(2_OVER_PI));
  double t = gm_fma(-kd, GMC(PIO2_1), x); /* exact (cancellation) */
  double ph = kd * GMC(PIO2_2);
  double pl = gm_fma(kd, GMC(PIO2_2), -ph); /* ph + pl == kd*PIO2_2 */
  double nph = -ph;
  double rh = t + nph; /* TwoSum(t, -ph) */
  double bb = rh - t;
  double e = (t - (rh - bb)) + (nph - bb);
  double lo = (e - pl) - kd * GMC(PIO2_3);
  double r0 = rh + lo;
  *rl = (rh - r0) + lo;
  *r = r0;
  return (int)((int64_t)kd & 3); /* |kd| < 2^50: the conversion is in range */
}

/* x - k*pi/2 as a double-double (r, rl) for every finite x; returns k mod 4 */
GM_HD int gm_rem_pio2(double x, double* r, double* rl) {
  if ((gm_d2u(x) & GM_ABS_MASK) >= GM_REM_PIO2_LARGE) {
    const GmRem R = gm_rem_pio2_large(x);
    *r = R.r;
    *rl = R.rl;
    return R.q;
  }
  return gm_rem_pio2_small(x, r, rl);
}

/* sin(x + y), |x| <~ pi/4, y a tail */
GM_HD double gm_ksin(double x, double y) {
  double z = x * x;
  double v = z * x;
  double p = GMC(SIN_C6);
  p = gm_fma(p, z, GMC(SIN_C5));
  p = gm_fma(p, z, GMC(SIN_C4));
  p = gm_fma(p, z, GMC(SIN_C3));
  p = gm_fma(p, z, GMC(SIN_C2));
  p = gm_fma(p, z, GMC(SIN_C1));
  return x - ((z * (0.5 * y - v * p) - y) - v * GMC(SIN_C0));
}

/* cos(x + y), |x| <~ pi/4, y a tail */
GM_HD double gm_kcos(double x, double y) {
  double z = x * x;
  double p = GMC(COS_C6);
  p = gm_fma(p, z, GMC(COS_C5));
  p = gm_fma(p, z, GMC(COS_C4));
  p = gm_fma(p, z, GMC(COS_C3));
  p = gm_fma(p, z, GMC(COS_C2));
  p = gm_fma(p, z, GMC(COS_C1));
  p = gm_fma(p, z, GMC(COS_C0));
  double hz = 0.5 * z;
  double w = 1.0 - hz;
  return w + (((1.0 - w) - hz) + (z * (z * p) - x * y));
}

/* sin and cos of x = k pi/2 + r + rl from the reduced argument and q = k mod 4 */
GM_HD void gm_sincos_reduced(double r, double rl, int q, double* s, double* c) {
  double ks = gm_ksin(r, rl);
  double kc = gm_kcos(r, rl);
  /* quadrant: q = 0 (s, c) | 1 (c, -s) | 2 (-s, -c) | 3 (-c, s); selects instead of a four-way branch */
  double ss = (q & 1) ? kc : ks;
  double cc = (q & 1) ? ks : kc;
  *s = (q & 2) ? -ss : ss;
  *c = ((q + 1) & 2) ? -cc : cc;
}

/* sin and cos for |x| >= GM_REM_PIO2_LARGE.  Inline, not a call: in the hot path (rotq_part) a call made the NLP
 * kernels spill more (-Xptxas -v: k_residuals 604 -> 636 bytes of spill loads) and the bench step slower than the
 * inlined form.  Inlined, the branch still costs +0.45 % of the bench step and changes the spills (stores / loads,
 * bytes): k_jacobian 308 / 552 -> 276 / 496 and k_residuals 508 / 604 -> 500 / 588 (fewer), the measurement-only
 * k_jacobian_heavy 36 / 56 -> 40 / 60 and k_jacobian_light 304 / 544 -> 320 / 576 (more).
 * profiles/r10_ptxas.txt, profiles/r10_bench.txt. */
typedef struct GmSinCos {
  double s, c;
} GmSinCos;
GM_HD GmSinCos gm_sincos_large(double x) {
  const GmRem R = gm_rem_pio2_large(x);
  GmSinCos v;
  gm_sincos_reduced(R.r, R.rl, R.q, &v.s, &v.c);
  return v;
}

/* gm_sincos_inl without the large-argument branch, for the hot-path callers whose argument is an atan2 result or
 * half of one (|x| <= pi): one copy of the large path fewer in each, which the bench step measured
 * (profiles/r10_bench.txt).  For |x| < GM_REM_PIO2_LARGE the same bits as gm_sincos_inl; from there on (and for inf
 * and NaN) NaN -- the one test that caught inf / NaN before, with a lower bound, so that gm_rem_pio2_small never sees
 * an argument whose k it cannot convert. */
GM_HD_INL void gm_sincos_small_inl(double x, double* s, double* c) {
  uint64_t ax = gm_d2u(x) & GM_ABS_MASK;
  if (ax >= GM_REM_PIO2_LARGE) { /* outside the domain, inf or nan */
    *s = gm_nan();
    *c = gm_nan();
    return;
  }
  double r = x, rl = 0.0;
  int q = 0;
  if (ax > 0x3fe921fb54442d18ull) /* |x| > pi/4 */
    q = gm_rem_pio2_small(x, &r, &rl);
  gm_sincos_reduced(r, rl, q, s, c);
}

GM_HD_INL void gm_sincos_inl(double x, double* s, double* c) {
  uint64_t ax = gm_d2u(x) & GM_ABS_MASK;
  if (ax >= GM_INF_BITS) { /* inf or nan */
    *s = gm_nan();
    *c = gm_nan();
    return;
  }
  if (ax >= GM_REM_PIO2_LARGE) {
    const GmSinCos v = gm_sincos_large(x);
    *s = v.s;
    *c = v.c;
    return;
  }
  double r = x, rl = 0.0;
  int q = 0;
  if (ax > 0x3fe921fb54442d18ull) /* |x| > pi/4 */
    q = gm_rem_pio2_small(x, &r, &rl);
  gm_sincos_reduced(r, rl, q, s, c);
}
GM_HD_CALL void gm_sincos(double x, double* s, double* c) { gm_sincos_inl(x, s, c); }

GM_HD double gm_sin(double x) {
  double s, c;
  gm_sincos(x, &s, &c);
  return s;
}

GM_HD double gm_cos(double x) {
  double s, c;
  gm_sincos(x, &s, &c);
  return c;
}

GM_HD_CALL double gm_tan(double x) {
  uint64_t ax = gm_d2u(x) & GM_ABS_MASK;
  if (ax >= GM_INF_BITS) return gm_nan();
  double r = x, rl = 0.0;
  int q = 0;
  if (ax > 0x3fe921fb54442d18ull) q = gm_rem_pio2(x, &r, &rl);
  double ks = gm_ksin(r, rl);
  double kc = gm_kcos(r, rl);
  return (q & 1) ? -kc / ks : ks / kc;
}

/* ---- atan / atan2 / asin / acos --------------------------------------- */

GM_HD double gm_atan_poly(double z) { /* (t - atan t)/t^3, z = t^2 <= (7/16)^2 */
  double p = GMC(ATAN_C13);
  p = gm_fma(p, z, GMC(ATAN_C12));
  p = gm_fma(p, z, GMC(ATAN_C11));
  p = gm_fma(p, z, GMC(ATAN_C10));
  p = gm_fma(p, z, GMC(ATAN_C9));
  p = gm_fma(p, z, GMC(ATAN_C8));
  p = gm_fma(p, z, GMC(ATAN_C7));
  p = gm_fma(p, z, GMC(ATAN_C6));
  p = gm_fma(p, z, GMC(ATAN_C5));
  p = gm_fma(p, z, GMC(ATAN_C4));
  p = gm_fma(p, z, GMC(ATAN_C3));
  p = gm_fma(p, z, GMC(ATAN_C2));
  p = gm_fma(p, z, GMC(ATAN_C1));
  p = gm_fma(p, z, GMC(ATAN_C0));
  return p;
}

/* atan(a) for 2^-27 <= a < 2^66 (the range reduction of gm_atan without its special cases) */
GM_HD double gm_atan_core(double a) {
  double t, hi, lo;
  if (a < 0.4375) {
    double z = a * a;
    return a - a * (z * gm_atan_poly(z));
  } else if (a < 0.6875) {
    t = gm_div(2.0 * a - 1.0, 2.0 + a);
    hi = GMC(ATAN_05_HI);
    lo = GMC(ATAN_05_LO);
  } else if (a < 1.1875) {
    t = gm_div(a - 1.0, a + 1.0);
    hi = GMC(ATAN_10_HI);
    lo = GMC(ATAN_10_LO);
  } else if (a < 2.4375) {
    t = gm_div(a - 1.5, 1.0 + 1.5 * a);
    hi = GMC(ATAN_15_HI);
    lo = GMC(ATAN_15_LO);
  } else {
    t = gm_div(-1.0, a);
    hi = GMC(ATAN_INF_HI);
    lo = GMC(ATAN_INF_LO);
  }
  double z = t * t;
  double corr = t * (z * gm_atan_poly(z)); /* t - atan(t) */
  return hi - ((corr - lo) - t);
}

GM_HD double gm_atan(double x) {
  uint64_t ux = gm_d2u(x);
  uint64_t ax = ux & GM_ABS_MASK;
  if (ax > GM_INF_BITS) return x + x; /* nan */
  double a = gm_u2d(ax);
  if (ax >= 0x4410000000000000ull) /* |x| >= 2^66 */
    return gm_copysign(GMC(ATAN_INF_HI), x);
  if (ax < 0x3e40000000000000ull) /* |x| < 2^-27 */
    return x;
  if (a < 0.4375) { /* the odd polynomial on the signed argument, as before */
    double z = x * x;
    return x - x * (z * gm_atan_poly(z));
  }
  double res = gm_atan_core(a);
  return (ux & GM_SIGN_MASK) ? -res : res;
}

/* every special case of atan2: zeros, infinities, NaN, extreme quotients */
GM_HD_CALL double gm_atan2_slow(double y, double x) {
  if (gm_isnan(x) || gm_isnan(y)) return x + y;
  uint64_t ux = gm_d2u(x), uy = gm_d2u(y);
  uint64_t ax = ux & GM_ABS_MASK, ay = uy & GM_ABS_MASK;
  int m = (int)(uy >> 63) | ((int)(ux >> 63) << 1); /* 2*sign(x) + sign(y) */
  const double pi = GMC(PI_HI), pi_lo = GMC(PI_LO);
  if (ay == 0) {
    switch (m) {
      case 0:
      case 1: return y; /* atan(+-0, +anything) = +-0 */
      case 2: return pi;
      default: return -pi;
    }
  }
  if (ax == 0) return (m & 1) ? -GMC(ATAN_INF_HI) : GMC(ATAN_INF_HI);
  if (ax == GM_INF_BITS) {
    if (ay == GM_INF_BITS) {
      switch (m) {
        case 0: return GMC(ATAN_10_HI);
        case 1: return -GMC(ATAN_10_HI);
        case 2: return 3.0 * GMC(ATAN_10_HI);
        default: return -3.0 * GMC(ATAN_10_HI);
      }
    } else {
      switch (m) {
        case 0: return 0.0;
        case 1: return -0.0;
        case 2: return pi;
        default: return -pi;
      }
    }
  }
  if (ay == GM_INF_BITS) return (m & 1) ? -GMC(ATAN_INF_HI) : GMC(ATAN_INF_HI);

  int k = (int)(ay >> 52) - (int)(ax >> 52);
  double z;
  if (k > 64) { /* |y/x| > 2^64 */
    z = GMC(ATAN_INF_HI) + 0.5 * pi_lo;
    m &= 1;
  } else if ((m & 2) && k < -64) { /* 0 > |y|/x > -2^-64 */
    z = 0.0;
  } else {
    z = gm_atan(gm_div(gm_u2d(ay), gm_u2d(ax)));
  }
  switch (m) {
    case 0: return z;
    case 1: return -z;
    case 2: return pi - (z - pi_lo);
    default: return (z - pi_lo) - pi;
  }
}

/* atan2: the common case -- both arguments normal numbers whose exponents differ by less than 26, so that the
 * quotient lies in [2^-27, 2^27] -- goes straight to the range reduction (two integer tests instead of the ladder
 * of special cases, which ncu r02a showed as the kernel's most expensive branches); everything else takes
 * gm_atan2_slow.  Same operations in the same order on either route. */
GM_HD_INL double gm_atan2_inl(double y, double x) {
  const uint64_t ux = gm_d2u(x), uy = gm_d2u(y);
  const uint32_t ex = (uint32_t)(ux >> 52) & 0x7ffu, ey = (uint32_t)(uy >> 52) & 0x7ffu;
  const int k = (int)ey - (int)ex;
  if (ex - 1u < 0x7feu - 1u && ey - 1u < 0x7feu - 1u && k > -26 && k < 26) {
    const double z = gm_atan_core(gm_div(gm_u2d(uy & GM_ABS_MASK), gm_u2d(ux & GM_ABS_MASK)));
    const double pi = GMC(PI_HI), pi_lo = GMC(PI_LO);
    const double zx = (ux >> 63) ? pi - (z - pi_lo) : z; /* x < 0: second / third quadrant */
    return (uy >> 63) ? -zx : zx;
  }
  return gm_atan2_slow(y, x);
}
GM_HD_CALL double gm_atan2(double y, double x) { return gm_atan2_inl(y, x); }

GM_HD double gm_acos(double x) {
  if (gm_isnan(x)) return x + x;
  if (gm_fabs(x) > 1.0) return gm_nan();
  double y = gm_sqrt((1.0 - x) * (1.0 + x));
  return gm_atan2(y, x);
}

GM_HD double gm_asin(double x) {
  if (gm_isnan(x)) return x + x;
  if (gm_fabs(x) > 1.0) return gm_nan();
  double c = gm_sqrt((1.0 - x) * (1.0 + x));
  return gm_atan2(x, c);
}

/* ---- exp / pow -------------------------------------------------------- */

/* y * 2^k for y in [0.5, 2) */
GM_HD double gm_scale2(double y, int k) {
  if (k > 1023) {
    y *= 0x1p1023;
    k -= 1023;
    if (k > 1023) k = 1023;
  } else if (k < -1022) {
    y *= 0x1p-1000;
    k += 1000;
    if (k < -1022) k = -1022;
  }
  return y * gm_u2d((uint64_t)(k + 1023) << 52);
}

/* exp(x + xl), |xl| << |x| */
GM_HD_INL double gm_exp_dd_inl(double x, double xl) {
  if (gm_isnan(x)) return x + x;
  if (x > 709.782712893384) return gm_inf();
  if (x < -745.2) return 0.0;
  double kd = gm_rint(x * GMC(INV_LN2));
  double r = gm_fma(-kd, GMC(LN2_HI), x); /* exact */
  double lo = gm_fma(-kd, GMC(LN2_LO), xl);
  double rr = r + lo;
  double rl = (r - rr) + lo;
  double q = GMC(EXP_C12);
  q = gm_fma(q, rr, GMC(EXP_C11));
  q = gm_fma(q, rr, GMC(EXP_C10));
  q = gm_fma(q, rr, GMC(EXP_C9));
  q = gm_fma(q, rr, GMC(EXP_C8));
  q = gm_fma(q, rr, GMC(EXP_C7));
  q = gm_fma(q, rr, GMC(EXP_C6));
  q = gm_fma(q, rr, GMC(EXP_C5));
  q = gm_fma(q, rr, GMC(EXP_C4));
  q = gm_fma(q, rr, GMC(EXP_C3));
  q = gm_fma(q, rr, GMC(EXP_C2));
  q = gm_fma(q, rr, GMC(EXP_C1));
  q = gm_fma(q, rr, GMC(EXP_C0));
  double p = (rr * rr) * q;
  double s = rr + (p + gm_fma(rl, rr, rl));
  double y = 1.0 + s;
  return gm_scale2(y, (int)kd); /* the guards above keep |kd| <= 1076: the conversion is in range */
}

GM_HD_CALL double gm_exp_dd(double x, double xl) { return gm_exp_dd_inl(x, xl); }

GM_HD double gm_exp(double x) { return gm_exp_dd(x, 0.0); }
GM_HD_INL double gm_exp_inl(double x) { return gm_exp_dd_inl(x, 0.0); }

/* log(x) as a double-double (hi, lo), x finite > 0 (subnormals handled) */
GM_HD void gm_log_dd(double x, double* hi, double* lo) {
  uint64_t ux = gm_d2u(x);
  int k = 0;
  if (ux < 0x0010000000000000ull) { /* subnormal */
    x *= 0x1p54;
    ux = gm_d2u(x);
    k = -54;
  }
  k += (int)(ux >> 52) - 1023;
  uint64_t man = ux & 0x000fffffffffffffull;
  double m;
  if (man > 0x6a09e667f3bcdull) { /* m > sqrt(2): use m/2 */
    m = gm_u2d(man | 0x3fe0000000000000ull);
    k += 1;
  } else {
    m = gm_u2d(man | 0x3ff0000000000000ull);
  }
  double f = m - 1.0; /* exact */
  double dh = 2.0 + f;
  double dl = (2.0 - dh) + f;
  double sh = f / dh;
  double rem = gm_fma(-sh, dh, f);
  rem = gm_fma(-sh, dl, rem);
  double sl = rem / dh;
  double z = sh * sh;
  double L = GMC(LOG_C12);
  L = gm_fma(L, z, GMC(LOG_C11));
  L = gm_fma(L, z, GMC(LOG_C10));
  L = gm_fma(L, z, GMC(LOG_C9));
  L = gm_fma(L, z, GMC(LOG_C8));
  L = gm_fma(L, z, GMC(LOG_C7));
  L = gm_fma(L, z, GMC(LOG_C6));
  L = gm_fma(L, z, GMC(LOG_C5));
  L = gm_fma(L, z, GMC(LOG_C4));
  L = gm_fma(L, z, GMC(LOG_C3));
  L = gm_fma(L, z, GMC(LOG_C2));
  L = gm_fma(L, z, GMC(LOG_C1));
  L = gm_fma(L, z, GMC(LOG_C0));
  double T = (sh * z) * L;      /* 2*atanh(sh) - 2*sh */
  T = gm_fma(2.0 * z, sl, T);   /* first-order effect of sl on the tail */
  double A = 2.0 * sh;
  double al = gm_fma(2.0, sl, T);
  double kd = (double)k;
  double kh = kd * GMC(LN2_HI);
  double kl = gm_fma(kd, GMC(LN2_HI), -kh);
  kl = gm_fma(kd, GMC(LN2_LO), kl);
  double h = kh + A; /* TwoSum */
  double bb = h - kh;
  double e = (kh - (h - bb)) + (A - bb);
  double l = e + (kl + al);
  double h2 = h + l;
  *lo = (h - h2) + l;
  *hi = h2;
}

GM_HD double gm_log(double x) {
  if (gm_isnan(x)) return x + x;
  if (x < 0.0) return gm_nan();
  if (x == 0.0) return -gm_inf();
  if (gm_d2u(x) == GM_INF_BITS) return x;
  double h, l;
  gm_log_dd(x, &h, &l);
  return h;
}

GM_HD int gm_is_int(double y) { /* |y| < 2^51 assumed for the rint trick */
  double a = gm_fabs(y);
  if (a >= 0x1p53) return 1;
  if (a >= 0x1p51) { /* few fractional bits left: test directly */
    uint64_t u = gm_d2u(a);
    int e = (int)(u >> 52) - 1023;
    uint64_t frac_mask = (1ull << (52 - e)) - 1ull;
    return (u & frac_mask) == 0;
  }
  return gm_rint(a) == a;
}

GM_HD int gm_is_odd_int(double y) {
  double a = gm_fabs(y);
  if (a >= 0x1p53) return 0;
  if (!gm_is_int(y)) return 0;
  double h = a * 0.5;
  return !gm_is_int(h);
}

/* every special case of pow: zero / one / infinite / NaN / negative arguments */
GM_HD_CALL double gm_pow_slow(double x, double y) {
  if (y == 0.0) return 1.0;
  if (x == 1.0) return 1.0;
  if (gm_isnan(x) || gm_isnan(y)) return x + y;
  uint64_t ax = gm_d2u(x) & GM_ABS_MASK, ay = gm_d2u(y) & GM_ABS_MASK;
  double sgn = 1.0;
  if (ay == GM_INF_BITS) {
    double a = gm_u2d(ax);
    if (a == 1.0) return 1.0;
    return ((a > 1.0) == (y > 0.0)) ? gm_inf() : 0.0;
  }
  if (gm_d2u(x) & GM_SIGN_MASK) { /* negative base (or -0) */
    if (ax == 0) {
      int odd = gm_is_odd_int(y);
      if (y > 0.0) return odd ? -0.0 : 0.0;
      return odd ? -gm_inf() : gm_inf();
    }
    if (ax == GM_INF_BITS) { /* C99 F.9.4.4: -inf to a power that is not an odd integer is +inf or +0, not NaN */
      const int odd = gm_is_odd_int(y);
      if (y > 0.0) return odd ? -gm_inf() : gm_inf();
      return odd ? -0.0 : 0.0;
    }
    if (!gm_is_int(y)) return gm_nan();
    if (gm_is_odd_int(y)) sgn = -1.0;
    x = gm_u2d(ax);
  }
  if (ax == 0) return (y > 0.0) ? 0.0 : gm_inf();
  if (ax == GM_INF_BITS) return (y > 0.0) ? sgn * gm_inf() : sgn * 0.0;
  double lh, ll;
  gm_log_dd(x, &lh, &ll);
  double ph = y * lh;
  double pl = gm_fma(y, lh, -ph);
  pl = gm_fma(y, ll, pl);
  return sgn * gm_exp_dd(ph, pl);
}

/* pow: a positive normal base other than 1 and a finite non-zero exponent (two integer tests) go straight to
 * exp(y log x) in double-double; everything else takes gm_pow_slow.  Same operations on either route. */
GM_HD_INL double gm_pow_inl(double x, double y) {
  const uint64_t ux = gm_d2u(x), uy = gm_d2u(y);
  const uint32_t ex = (uint32_t)(ux >> 52), ey = (uint32_t)(uy >> 52) & 0x7ffu; /* ex includes the sign bit */
  if (ex - 1u < 0x7feu - 1u && ey != 0x7ffu && (uy << 1) != 0 && ux != 0x3ff0000000000000ull) {
    double lh, ll;
    gm_log_dd(x, &lh, &ll);
    double ph = y * lh;
    double pl = gm_fma(y, lh, -ph);
    pl = gm_fma(y, ll, pl);
    return gm_exp_dd_inl(ph, pl);
  }
  return gm_pow_slow(x, y);
}
GM_HD_CALL double gm_pow(double x, double y) { return gm_pow_inl(x, y); }

#endif /* GELATO_B200_GMATH_H_ */
