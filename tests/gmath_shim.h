/* The entry points of the gmath.h test shims, written once: tests/gmath_host_shim.c (g++ / gcc) and
 * tests/gmath_device_shim.cu (nvcc, one kernel per entry point) both expand GMATH_SHIM_ENTRIES, so the two builds
 * export the same set under the same names (gmt_<name>).  Four shapes:
 *   U(name, expr)   one input a, one output
 *   B(name, expr)   two inputs a, b, one output
 *   T(name, expr)   three inputs a, b, c, one output
 *   U2(name, stmt)  one input a, two outputs y0, y1 */
#ifndef GELATO_B200_TESTS_GMATH_SHIM_H_
#define GELATO_B200_TESTS_GMATH_SHIM_H_

#include "../gelato_b200/csrc/gmath.h"

GM_HD double gms_sin_inl(double x) {
  double s, c;
  gm_sincos_inl(x, &s, &c);
  return s;
}
GM_HD double gms_cos_inl(double x) {
  double s, c;
  gm_sincos_inl(x, &s, &c);
  return c;
}
GM_HD void gms_rcp(double d, double* r, double* ok) {
  const GmRcp R = gm_rcp(d);
  *r = R.r;
  *ok = R.ok ? 1.0 : 0.0;
}

#define GMATH_SHIM_ENTRIES(U, B, T, U2)          \
  U(sin, gm_sin(a))                              \
  U(sin_inl, gms_sin_inl(a))                     \
  U(cos, gm_cos(a))                              \
  U(cos_inl, gms_cos_inl(a))                     \
  U2(sincos, gm_sincos(a, &y0, &y1))             \
  U2(sincos_inl, gm_sincos_inl(a, &y0, &y1))     \
  U2(sincos_small_inl, gm_sincos_small_inl(a, &y0, &y1)) \
  U(tan, gm_tan(a))                              \
  U(atan, gm_atan(a))                            \
  B(atan2, gm_atan2(a, b))                       \
  B(atan2_inl, gm_atan2_inl(a, b))               \
  B(atan2_slow, gm_atan2_slow(a, b))             \
  U(asin, gm_asin(a))                            \
  U(acos, gm_acos(a))                            \
  U(exp, gm_exp(a))                              \
  U(exp_inl, gm_exp_inl(a))                      \
  B(exp_dd, gm_exp_dd(a, b))                     \
  U2(log_dd, gm_log_dd(a, &y0, &y1))             \
  U(log, gm_log(a))                              \
  B(pow, gm_pow(a, b))                           \
  B(pow_inl, gm_pow_inl(a, b))                   \
  B(pow_slow, gm_pow_slow(a, b))                 \
  U2(rcp, gms_rcp(a, &y0, &y1))                  \
  B(div_by, gm_div_by(a, gm_rcp(b)))             \
  U(sqrt, gm_sqrt(a))                            \
  T(fma, gm_fma(a, b, c))

#endif /* GELATO_B200_TESTS_GMATH_SHIM_H_ */
