/* Host-side export of gmath.h for tests/test_gmath.py and tests/test_gmath_device.py (accuracy vs mpmath, and the
 * host side of device == host).  Built by those tests with: gcc -O2 -ffp-contract=off -mfma -shared -fPIC */
#include "gmath_shim.h"

#define U(name, expr) \
  void gmt_##name(const double* x, double* y, int n) { for (int i = 0; i < n; i++) { const double a = x[i]; y[i] = expr; } }
#define B(name, expr)                                                       \
  void gmt_##name(const double* x, const double* w, double* y, int n) {     \
    for (int i = 0; i < n; i++) { const double a = x[i], b = w[i]; y[i] = expr; } \
  }
#define T(name, expr)                                                                        \
  void gmt_##name(const double* x, const double* w, const double* v, double* y, int n) {    \
    for (int i = 0; i < n; i++) { const double a = x[i], b = w[i], c = v[i]; y[i] = expr; } \
  }
#define U2(name, stmt)                                              \
  void gmt_##name(const double* x, double* y, double* z, int n) {   \
    for (int i = 0; i < n; i++) {                                   \
      const double a = x[i];                                        \
      double y0, y1;                                                \
      stmt;                                                         \
      y[i] = y0;                                                    \
      z[i] = y1;                                                    \
    }                                                               \
  }
GMATH_SHIM_ENTRIES(U, B, T, U2)
