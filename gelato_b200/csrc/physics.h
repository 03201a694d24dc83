/* physics.h -- the 3-DoF launch-vehicle physics leaves, written for GPU threads
 * that each evaluate one (node x perturbation column) or a shareable part of it
 * (pos_part / rotq_part / per-column remainder: see "the air right-hand side in
 * three parts" below and jobs.h).
 *
 * Each function states which reference routine it replaces.  Values are
 * bit-identical to the reference's formulas evaluated in IEEE binary64 with
 * unfused multiply-add (the reference is built for baseline x86-64, no FMA:
 * /root/reference/CMakeLists.txt:8,41), with the elementary functions taken
 * from gmath.h (DESIGN.md H1).  Compile with nvcc -fmad=false.
 *
 * Unlike the reference, common sub-expressions are evaluated once per thread:
 * one geodetic conversion for the altitude, one US-76 layer lookup shared by
 * temperature / pressure / density / speed of sound, one sincos of the Earth
 * rotation angle shared by every frame rotation
 * (reference recomputes them: pybind_dynamics.cpp:42-68 calls ecef2geodetic
 * twice, Air::us76_params five times, cos/sin(omega t) ~10 times).
 *
 * The header is host+device so the very same code can be stepped through by
 * the host emulator in tests/emu (test harness only; the product library only
 * ever launches it on the GPU).
 */
#ifndef GELATO_B200_PHYSICS_H_
#define GELATO_B200_PHYSICS_H_

#include "gmath.h"

#define P_HD GM_HD
#define P_HD_CALL GM_HD_CALL

#define P_PI 3.14159265358979323846
#define P_MU 3.986004418e14
#define P_OMEGA 7.2921151467e-5
#define P_RA 6378137.0
#define P_F (1.0 / 298.257223563)
#define P_RB (P_RA * (1.0 - P_F))
#define P_E2 ((P_RA * P_RA - P_RB * P_RB) / P_RA / P_RA)
#define P_EP2 ((P_RA * P_RA - P_RB * P_RB) / P_RB / P_RB)

struct Vec3 {
  double x, y, z;
};
struct Quat {
  double w, x, y, z;
};

P_HD Vec3 v3(double x, double y, double z) {
  Vec3 r;
  r.x = x; r.y = y; r.z = z;
  return r;
}
P_HD Quat q4(double w, double x, double y, double z) {
  Quat r;
  r.w = w; r.x = x; r.y = y; r.z = z;
  return r;
}

/* Eigen-style 3-vector reductions, order (a0 + a1) + a2 (see oracle_leaves.cpp) */
P_HD double dot3(Vec3 a, Vec3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
P_HD double norm3(Vec3 a) { return gm_sqrt(dot3(a, a)); }
P_HD Vec3 cross3(Vec3 a, Vec3 b) {
  return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
P_HD Vec3 sub3(Vec3 a, Vec3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
P_HD Vec3 add3(Vec3 a, Vec3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
P_HD Vec3 scale3(double s, Vec3 a) { return v3(s * a.x, s * a.y, s * a.z); }
P_HD Vec3 div3(Vec3 a, double s) {
  const GmRcp R = gm_rcp(s); /* one reciprocal for the three quotients (gmath.h: gm_div_by is the IEEE quotient) */
  return v3(gm_div_by(a.x, R), gm_div_by(a.y, R), gm_div_by(a.z, R));
}
P_HD Vec3 normalized3(Vec3 a) { /* Eigen normalized() */
  double z = dot3(a, a);
  if (z > 0.0) return div3(a, gm_sqrt(z));
  return a;
}

/* wrapper_coordinate.hpp:50-57 quatmult */
P_HD Quat quatmult(Quat q, Quat p) {
  return q4(q.w * p.w - q.x * p.x - q.y * p.y - q.z * p.z,
            q.w * p.x + q.x * p.w + q.y * p.z - q.z * p.y,
            q.w * p.y - q.x * p.z + q.y * p.w + q.z * p.x,
            q.w * p.z + q.x * p.y - q.y * p.x + q.z * p.w);
}
/* Eigen::Quaterniond operator* (Coordinate.cpp:104-106) */
P_HD Quat eigen_quat_prod(Quat a, Quat b) {
  return q4(a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z,
            a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
            a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z,
            a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x);
}
P_HD Quat quatconj(Quat q) { return q4(q.w, -q.x, -q.y, -q.z); }
/* wrapper_coordinate.hpp:70-78 quatrot */
P_HD Vec3 quatrot(Quat q, Vec3 v) {
  Quat vq = q4(0.0, v.x, v.y, v.z);
  Quat r = quatmult(quatconj(q), quatmult(vq, q));
  return v3(r.x, r.y, r.z);
}

/* ---- geodesy (Earth.cpp:49-61) ------------------------------------------ */
struct Geodetic {
  double lat, lon, alt; /* radians, radians, metres */
};
/* WANT: bit0 altitude, bit1 longitude (latitude is always produced).  HOT: the elementary functions inlined
 * (gmath.h: gm_xxx_inl) -- for the two callers that are the Jacobian kernel's long items.  The sines and cosines here
 * are of atan2 results (|x| <= pi): gm_sincos_small_inl. */
template <int WANT, bool HOT = false>
P_HD Geodetic ecef2geodetic(Vec3 r) {
  Geodetic g;
  double p = gm_sqrt(r.x * r.x + r.y * r.y);
  double theta = HOT ? gm_atan2_inl(r.z * P_RA, p * P_RB) : gm_atan2(r.z * P_RA, p * P_RB);
  double st, ct;
  if (HOT) gm_sincos_small_inl(theta, &st, &ct);
  else gm_sincos(theta, &st, &ct);
  const double ny = r.z + P_EP2 * P_RB * (st * st * st), nx = p - P_E2 * P_RA * (ct * ct * ct);
  g.lat = HOT ? gm_atan2_inl(ny, nx) : gm_atan2(ny, nx);
  g.lon = 0.0;
  g.alt = 0.0;
  if (WANT & 2) g.lon = HOT ? gm_atan2_inl(r.y, r.x) : gm_atan2(r.y, r.x);
  if (WANT & 1) {
    double sl, cl;
    if (HOT) gm_sincos_small_inl(g.lat, &sl, &cl);
    else gm_sincos(g.lat, &sl, &cl);
    double N = gm_div(P_RA, gm_sqrt(1.0 - P_E2 * sl * sl));
    g.alt = gm_div(p, cl) - N;
  }
  return g;
}

/* Coordinate.cpp:41-59 with cos/sin(omega t) supplied */
P_HD Vec3 rot_ecef2eci(Vec3 a, double c, double s) { return v3(a.x * c - a.y * s, a.x * s + a.y * c, a.z); }
P_HD Vec3 rot_eci2ecef(Vec3 a, double c, double s) { return v3(a.x * c + a.y * s, -a.x * s + a.y * c, a.z); }

/* Coordinate.cpp:69-73 vel_eci2ecef */
P_HD Vec3 vel_eci2ecef_cs(Vec3 vel, Vec3 pos, double c, double s) {
  Vec3 w = v3(0.0, 0.0, P_OMEGA);
  return rot_eci2ecef(sub3(vel, cross3(w, pos)), c, s);
}
/* Coordinate.cpp:61-67 vel_ecef2eci */
P_HD Vec3 vel_ecef2eci_cs(Vec3 vel_ecef, Vec3 pos_ecef, double c, double s) {
  Vec3 pos_eci = rot_ecef2eci(pos_ecef, c, s);
  Vec3 vg = rot_ecef2eci(vel_ecef, c, s);
  Vec3 w = v3(0.0, 0.0, P_OMEGA);
  return add3(vg, cross3(w, pos_eci));
}

/* Coordinate.cpp:85-98 quat_ecef2ned from geodetic lat/lon */
template <bool HOT = false>
P_HD Quat quat_ecef2ned_ll(double lat, double lon) {
  double s_hl, c_hl, s_hp, c_hp;
  if (HOT) {
    gm_sincos_small_inl(lon / 2.0, &s_hl, &c_hl);
    gm_sincos_small_inl(lat / 2.0, &s_hp, &c_hp);
  } else {
    gm_sincos(lon / 2.0, &s_hl, &c_hl);
    gm_sincos(lat / 2.0, &s_hp, &c_hp);
  }
  const GmRcp r2 = gm_rcp(gm_sqrt(2.0)); /* a compile-time constant and its reciprocal */
  return q4(gm_div_by(c_hl * (c_hp - s_hp), r2), gm_div_by(s_hl * (c_hp + s_hp), r2), gm_div_by(-c_hl * (c_hp + s_hp), r2),
            gm_div_by(s_hl * (c_hp - s_hp), r2));
}

/* Coordinate.cpp:104-110 quat_ned2eci(pos_eci, t); c,s = cos/sin(omega t) */
template <bool HOT = false>
P_HD Quat quat_ned2eci_cs(Vec3 pos_eci, double wt, double c, double s) {
  double sh, ch;
  if (HOT) gm_sincos_inl(wt / 2.0, &sh, &ch);
  else gm_sincos(wt / 2.0, &sh, &ch);
  Quat q_eci2ecef = q4(ch, 0.0, 0.0, sh);
  Geodetic g = ecef2geodetic<2, HOT>(rot_eci2ecef(pos_eci, c, s));
  Quat q = eigen_quat_prod(q_eci2ecef, quat_ecef2ned_ll<HOT>(g.lat, g.lon));
  return quatconj(q);
}

/* ---- gravity (gravity.cpp:11-57) ---------------------------------------- */
P_HD Vec3 gravity_eci(Vec3 pos) {
  const double a = 6378137.0, one_f = 298.257223563, mu = 3.986004418e14;
  const double barC20 = -0.484165371736e-3;
  const double f = 1.0 / one_f;
  const double b = a * (1.0 - f);
  double x = pos.x, y = pos.y, z = pos.z;
  double r = gm_sqrt(x * x + y * y + z * z);
  double irx, iry, irz;
  if (r == 0.0) {
    irx = iry = irz = 0.0;
  } else {
    const GmRcp Rr = gm_rcp(r);
    irx = gm_div_by(x, Rr);
    iry = gm_div_by(y, Rr);
    irz = gm_div_by(z, Rr);
  }
  double s5 = gm_sqrt(5.0);
  double barP20 = s5 * (3.0 * irz * irz - 1.0) * 0.5;
  double barP20d = s5 * 3.0 * irz;
  if (r < b) r = b;
  /* the reference writes a / r four times and mu / (r * r) twice (gravity.cpp:49-53); equal operands give
   * equal quotients, and (-mu) / d == -(mu / d) exactly, so each is divided once */
  const double a_r = gm_div(a, r), mu_r2 = gm_div(mu, r * r);
  double g_ir = -mu_r2 * (1.0 + barC20 * a_r * a_r * (3.0 * barP20 + irz * barP20d));
  double g_iz = mu_r2 * a_r * a_r * barC20 * barP20d;
  return v3(g_ir * irx, g_ir * iry, g_ir * irz + g_iz);
}

/* ---- US Standard Atmosphere 1976 (Air.cpp:28-111) ------------------------ */
struct AirState {
  double T, P, rho, a;
};

P_HD double geopotential_altitude(double z) {
  if (z < 86000.0) return gm_div(1.0 * (6356766.0 * z), 6356766.0 + z);
  return z;
}

/* One row of the US-76 layer table (Air.cpp:31-45) and what depends on that row only:
 * R = Rstar / M, the pressure exponent -g0 / Lmb / R (gradient layers) and g0 / R (isothermal layers).
 * They are constant expressions of the row -- the reference evaluates them again on every call
 * (Air.cpp:62-67, 93-97); here they are folded at compile time with the same IEEE divisions. */
struct Us76Layer {
  double Hb, Lmb, Tmb, Pb, R, expo, g0_R;
};
#define US76_ROW(hb_, l_, t_, p_, m_)                                                                          \
  { (hb_), (l_), (t_), (p_), 8314.32 / (m_), ((l_) != 0.0) ? -9.80665 / (l_) / (8314.32 / (m_)) : 0.0,         \
    9.80665 / (8314.32 / (m_)) }
#define US76_TABLE                                                                                             \
  {                                                                                                            \
    US76_ROW(0.0, -0.0065, 288.15, 101325.0, 28.9644), US76_ROW(11000.0, 0.0, 216.65, 22632.0, 28.9644),       \
    US76_ROW(20000.0, 0.001, 216.65, 5474.9, 28.9644), US76_ROW(32000.0, 0.0028, 228.65, 868.02, 28.9644),     \
    US76_ROW(47000.0, 0.0, 270.65, 110.91, 28.9644), US76_ROW(51000.0, -0.0028, 270.65, 66.939, 28.9644),      \
    US76_ROW(71000.0, -0.002, 214.65, 3.9564, 28.9644), US76_ROW(86000.0, 0.0, 186.8673, 0.37338, 28.9522),    \
    US76_ROW(91000.0, 0.0025, 186.8673, 0.15381, 28.89), US76_ROW(110000.0, 0.012, 240.0, 7.1042e-3, 27.27),   \
    US76_ROW(120000.0, 0.012, 360.0, 2.5382e-3, 26.20)                                                         \
  }
#if defined(__CUDACC__)
static __constant__ Us76Layer us76_table_dev[11] = US76_TABLE;
#endif
P_HD Us76Layer us76_layer(double h) {
  /* last layer whose base is <= h; layer 0 when h is below every base (Air.cpp:56-60): the bases ascend, so
   * that is a count of bases <= h -- ten compares and one indexed read of the row (the table sits in constant
   * memory on the device) instead of a ladder that rewrote seven doubles per rung */
  int k = 0;
  k += (h >= 11000.0); k += (h >= 20000.0); k += (h >= 32000.0); k += (h >= 47000.0); k += (h >= 51000.0);
  k += (h >= 71000.0); k += (h >= 86000.0); k += (h >= 91000.0); k += (h >= 110000.0); k += (h >= 120000.0);
#if defined(__CUDA_ARCH__)
  return us76_table_dev[k];
#else
  static const Us76Layer table[11] = US76_TABLE;
  return table[k];
#endif
}

/* want: bit0 pressure+density, bit1 speed of sound.  HOT: elementary functions inlined (see ecef2geodetic). */
template <bool HOT = false>
P_HD AirState us76(double h, int want) {
  const double r0 = 6356766.0;
  const Us76Layer L = us76_layer(h);
  const double Hb = L.Hb, Lmb = L.Lmb, Tmb = L.Tmb, Pb = L.Pb, R = L.R;
  AirState s;
  if (h <= 91000.0) {
    s.T = Tmb + Lmb * (h - Hb);
  } else if (h <= 110000.0) {
    const double Tc = 263.1905, A = -76.3232, a = -19942.9;
    s.T = Tc + A * gm_sqrt(1.0 - (h - 91000.0) * (h - 91000.0) / a / a);
  } else if (h <= 120000.0) {
    s.T = Tmb + Lmb * (h - Hb);
  } else {
    const double Tinf = 1000.0;
    double xi = (h - Hb) * (r0 + Hb) / (r0 + h);
    s.T = Tinf - (Tinf - Tmb) * gm_exp(-0.01875e-3 * xi);
  }
  s.P = 0.0;
  s.rho = 0.0;
  s.a = 0.0;
  if (want & 1) {
    if (gm_fabs(Lmb) > 1.0e-6) {
      const double base = gm_div(Tmb + Lmb * (h - Hb), Tmb);
      s.P = Pb * (HOT ? gm_pow_inl(base, L.expo) : gm_pow(base, L.expo)); /* -g0 / Lmb / R */
    } else {
      const double arg = gm_div(L.g0_R * (Hb - h), Tmb); /* g0 / R * (Hb - h) / Tmb */
      s.P = Pb * (HOT ? gm_exp_inl(arg) : gm_exp(arg));
    }
    s.rho = gm_div(gm_div(s.P, R), s.T);
  }
  if (want & 2) s.a = gm_sqrt(1.4 * R * s.T);
  return s;
}

/* ---- table interpolation (wrapper_utils.hpp:51-87) ----------------------- */
/* xp[i*stride], yp[i*stride]; lower_bound then idx-1 (x == xp[k] uses the interval
 * below; x == xp[0] would read xp[-1] in the reference -- defined here as interval 0,
 * like the oracle). */
/* interval of the table that x falls into: -1 below the first abscissa, -2 above the last, else idx */
P_HD int interp_interval(double x, const double* xp, int n, int stride) {
  if (x < xp[0]) return -1;
  if (x > xp[(n - 1) * stride]) return -2;
  /* lower_bound over a sorted table = number of entries below x; the tables have a
   * handful of rows, so a branch-free count beats a divergent binary search */
  int lo = 0;
  for (int i = 0; i < n; i++) lo += (xp[i * stride] < x) ? 1 : 0;
  int idx = lo - 1;
  if (idx < 0) idx = 0;
  return idx;
}
P_HD double interp_at(int idx, double x, const double* xp, const double* yp, int n, int stride) {
  if (idx == -1) return yp[0];
  if (idx == -2) return yp[(n - 1) * stride];
  double x_lower = xp[idx * stride], x_upper = xp[(idx + 1) * stride];
  double y_lower = yp[idx * stride], y_upper = yp[(idx + 1) * stride];
  double alpha = gm_div(x - x_lower, x_upper - x_lower);
  return y_lower + alpha * (y_upper - y_lower);
}
P_HD double interp_table(double x, const double* xp, const double* yp, int n, int stride) {
  return interp_at(interp_interval(x, xp, n, stride), x, xp, yp, n, stride);
}

/* ---- numpy's statements of two operations the Python layers around the NLP use (output.h, initguess.h) ---- */
/* numpy.linalg.norm of a 3-vector: sqrt of a BLAS dot, fused multiply-adds in ascending index */
P_HD double np_norm3(Vec3 v) { return gm_sqrt(gm_fma(v.z, v.z, gm_fma(v.y, v.y, v.x * v.x))); }

/* numpy.interp for one abscissa (numpy/_core/src/multiarray/compiled_base.c): interval by comparison count (the
 * tables are short), slope * (x - xp[j]) + fp[j] */
P_HD double np_interp(double x, const double* xp, const double* fp, int n, int stride) {
  if (x <= xp[0]) return fp[0];
  if (x >= xp[(n - 1) * stride]) return fp[(n - 1) * stride];
  int j = -1;
  for (int i = 0; i < n; i++) j += (xp[i * stride] <= x) ? 1 : 0;
  const double slope = (fp[(j + 1) * stride] - fp[j * stride]) / (xp[(j + 1) * stride] - xp[j * stride]);
  double res = slope * (x - xp[j * stride]) + fp[j * stride];
  if (res != res) {
    res = slope * (x - xp[(j + 1) * stride]) + fp[(j + 1) * stride];
    if (res != res && fp[j * stride] == fp[(j + 1) * stride]) res = fp[j * stride];
  }
  return res;
}

/* ---- the air right-hand side in three parts -------------------------------
 * The finite-difference columns of one node share most of their work: the
 * position-only part (geodetic altitude, atmosphere, wind lookup, gravity) takes
 * only 5 distinct inputs over the 14 columns, the position+time part (NED frame,
 * wind in ECI axes) 7.  The kernels therefore evaluate
 *     pos_part(pos)            once per distinct position,
 *     rotq_part(pos, t)        once per distinct (position, time), then rot_wind,
 *     a cheap per-column remainder,
 * with exactly the operations (and operation order) of the single-pass formulas in
 * pybind_dynamics.cpp:42-68 / wrapper_utils.hpp:89-193, so every column's bits
 * are what a full evaluation of that column gives. */
struct Tables {
  const double* wind; /* [n_wind][3]: altitude, wind_n, wind_e */
  int n_wind;
  const double* ca; /* [n_ca][2]: mach, CA */
  int n_ca;
};

enum { PP_WIND_N = 0, PP_WIND_E, PP_RHO, PP_PRESS, PP_SOUND, PP_GX, PP_GY, PP_GZ, PP_COLS };
enum { RP_COS = 0, RP_SIN, RP_WX, RP_WY, RP_WZ, RP_COLS };
enum { PW_GRAVITY = 1, PW_SOUND = 2 };

/* position-only part; pos dimensional (ECI fed to ecef2geodetic: quirk A.5-2).
 * pybind_dynamics.cpp:43-46,49,55,66 / wrapper_utils.hpp:93-95,164-172 */
P_HD_CALL void pos_part(double px, double py, double pz, const double* wind, int n_wind, int want, double* out) {
  Vec3 pos = v3(px, py, pz);
  Geodetic g = ecef2geodetic<1, true>(pos);
  double alt_gp = geopotential_altitude(g.alt);
  /* wind_ned interpolates both components at the same altitude (wrapper_utils.hpp:82-87): one interval search, one
   * interpolation weight -- the same quotient the two separate calls compute */
  const int iv = interp_interval(alt_gp, wind, n_wind, 3);
  if (iv < 0) {
    const int row = iv == -1 ? 0 : (n_wind - 1) * 3;
    out[PP_WIND_N] = wind[row + 1];
    out[PP_WIND_E] = wind[row + 2];
  } else {
    const double* w0 = wind + iv * 3;
    const double alpha = gm_div(alt_gp - w0[0], w0[3] - w0[0]);
    out[PP_WIND_N] = w0[1] + alpha * (w0[4] - w0[1]);
    out[PP_WIND_E] = w0[2] + alpha * (w0[5] - w0[2]);
  }
  AirState as = us76<true>(alt_gp, 1 | (want & PW_SOUND));
  out[PP_RHO] = as.rho;
  out[PP_PRESS] = as.P;
  out[PP_SOUND] = as.a;
  if (want & PW_GRAVITY) { /* otherwise the gravity fields are left to whoever computes them (jobs.h: dyn_air_phase) */
    const Vec3 gr = gravity_eci(pos);
    out[PP_GX] = gr.x;
    out[PP_GY] = gr.y;
    out[PP_GZ] = gr.z;
  }
}

/* position+time part, first half: cos/sin of the Earth-rotation angle and the
 * NED->ECI quaternion at that position and time.  t as the caller passes it (the
 * dynamics pass NON-dimensional node times -- quirk A.5-1 -- the aero constraints
 * pass seconds).  pybind_dynamics.cpp:48-51 */
enum { RQ_COS = 0, RQ_SIN, RQ_W, RQ_X, RQ_Y, RQ_Z, RQ_COLS };
P_HD_CALL void rotq_part(double px, double py, double pz, double t, double* out) {
  double wt = P_OMEGA * t;
  double s, c;
  gm_sincos_inl(wt, &s, &c);
  Quat q = quat_ned2eci_cs<true>(v3(px, py, pz), wt, c, s);
  out[RQ_COS] = c;
  out[RQ_SIN] = s;
  out[RQ_W] = q.w;
  out[RQ_X] = q.x;
  out[RQ_Y] = q.y;
  out[RQ_Z] = q.z;
}
/* second half: the wind of that altitude turned into ECI axes (pybind_dynamics.cpp:52) */
P_HD void rot_wind(const double* rq, double wind_n, double wind_e, double* out) {
  Vec3 wind_eci = quatrot(q4(rq[RQ_W], rq[RQ_X], rq[RQ_Y], rq[RQ_Z]), v3(wind_n, wind_e, 0.0));
  out[RP_COS] = rq[RQ_COS];
  out[RP_SIN] = rq[RQ_SIN];
  out[RP_WX] = wind_eci.x;
  out[RP_WY] = wind_eci.y;
  out[RP_WZ] = wind_eci.z;
}
P_HD void rot_part(double px, double py, double pz, double t, double wind_n, double wind_e, double* out) {
  double rq[RQ_COLS];
  rotq_part(px, py, pz, t, rq);
  rot_wind(rq, wind_n, wind_e, out);
}

/* air-relative velocity in ECI axes: pybind_dynamics.cpp:47,53 */
P_HD Vec3 air_velocity(Vec3 pos, Vec3 vel, const double* rp) {
  Vec3 vel_ecef = vel_eci2ecef_cs(vel, pos, rp[RP_COS], rp[RP_SIN]);
  return sub3(rot_ecef2eci(vel_ecef, rp[RP_COS], rp[RP_SIN]), v3(rp[RP_WX], rp[RP_WY], rp[RP_WZ]));
}

/* ---- dynamics right-hand sides (pybind_dynamics.cpp:30-106) -------------- */
struct SecParam {
  double thrust, massflow, ref_area, nozzle_area;
};
struct Units {
  double mass, pos, vel, u, t, dx;
};

/* dynamics_velocity, per-column remainder: acceleration / unit_vel.  mass_e / pos_e /
 * vel_e non-dimensional; pp = pos_part(pos_e*unit_pos), rp = rot_part(the same pos, t). */
P_HD Vec3 rhs_velocity_air_col(double mass_e, Vec3 pos_e, Vec3 vel_e, Quat q, const double* pp, const double* rp,
                               const SecParam& sp, const Units& un, const Tables& tb) {
  double mass = mass_e * un.mass;
  Vec3 pos = v3(pos_e.x * un.pos, pos_e.y * un.pos, pos_e.z * un.pos);
  Vec3 vel = v3(vel_e.x * un.vel, vel_e.y * un.vel, vel_e.z * un.vel);
  Vec3 va = air_velocity(pos, vel, rp);
  double vn = norm3(va);
  double mach = gm_div(vn, pp[PP_SOUND]);
  double ca = interp_table(mach, tb.ca, tb.ca + 1, tb.n_ca, 2);
  double k = 0.5 * pp[PP_RHO] * sp.ref_area * ca * vn;
  Vec3 aero = v3(k * -va.x, k * -va.y, k * -va.z);
  double thrust = sp.thrust - sp.nozzle_area * pp[PP_PRESS];
  Vec3 tdir = quatrot(quatconj(q), v3(1.0, 0.0, 0.0));
  Vec3 thr = scale3(thrust, tdir);
  const GmRcp Rm = gm_rcp(mass), Rv = gm_rcp(un.vel);
  return v3(gm_div_by(gm_div_by(thr.x + aero.x, Rm) + pp[PP_GX], Rv), gm_div_by(gm_div_by(thr.y + aero.y, Rm) + pp[PP_GY], Rv),
            gm_div_by(gm_div_by(thr.z + aero.z, Rm) + pp[PP_GZ], Rv));
}

/* dynamics_velocity in one pass (residual kernel: one evaluation per node) */
P_HD Vec3 rhs_velocity_air(double mass_e, Vec3 pos_e, Vec3 vel_e, Quat q, double t, const SecParam& sp,
                           const Units& un, const Tables& tb) {
  double pp[PP_COLS], rp[RP_COLS];
  double px = pos_e.x * un.pos, py = pos_e.y * un.pos, pz = pos_e.z * un.pos;
  pos_part(px, py, pz, tb.wind, tb.n_wind, PW_GRAVITY | PW_SOUND, pp);
  rot_part(px, py, pz, t, pp[PP_WIND_N], pp[PP_WIND_E], rp);
  return rhs_velocity_air_col(mass_e, pos_e, vel_e, q, pp, rp, sp, un, tb);
}

/* dynamics_velocity_NoAir; g = gravity_eci(pos_e*unit_pos) */
P_HD Vec3 rhs_velocity_noair_col(double mass_e, Quat q, Vec3 g, const SecParam& sp, const Units& un) {
  double mass = mass_e * un.mass;
  Vec3 tdir = quatrot(quatconj(q), v3(1.0, 0.0, 0.0));
  Vec3 thr = scale3(sp.thrust, tdir);
  const GmRcp Rm = gm_rcp(mass), Rv = gm_rcp(un.vel);
  return v3(gm_div_by(gm_div_by(thr.x, Rm) + g.x, Rv), gm_div_by(gm_div_by(thr.y, Rm) + g.y, Rv),
            gm_div_by(gm_div_by(thr.z, Rm) + g.z, Rv));
}
P_HD Vec3 rhs_velocity_noair(double mass_e, Vec3 pos_e, Quat q, const SecParam& sp, const Units& un) {
  Vec3 pos = v3(pos_e.x * un.pos, pos_e.y * un.pos, pos_e.z * un.pos);
  return rhs_velocity_noair_col(mass_e, q, gravity_eci(pos), sp, un);
}

/* dynamics_quaternion: 0.5 * q (x) (0, 0, u0, u1) * pi/180 */
P_HD Quat rhs_quaternion(Quat q, double u0_e, double u1_e, double unit_u) {
  double u0 = u0_e * unit_u, u1 = u1_e * unit_u;
  Quat om = q4(0.0 * P_PI / 180.0, 0.0 * P_PI / 180.0, u0 * P_PI / 180.0, u1 * P_PI / 180.0);
  Quat d = quatmult(q, om);
  return q4(0.5 * d.w, 0.5 * d.x, 0.5 * d.y, 0.5 * d.z);
}

/* ---- aero constraint leaves (wrapper_utils.hpp:89-111,163-193) ----------- */
/* kind: 0 angle of attack [rad], 1 dynamic pressure [Pa], 2 q*alpha [Pa rad].
 * pos / vel dimensional; pp / rp from pos_part / rot_part of the same position (t in seconds). */
P_HD double aero_quantity_col(int kind, Vec3 pos, Vec3 vel, Quat q, const double* pp, const double* rp) {
  Vec3 va = air_velocity(pos, vel, rp);
  double alpha = 0.0, dynp = 0.0;
  if (kind != 1) {
    Vec3 tdir = quatrot(quatconj(q), v3(1.0, 0.0, 0.0));
    Vec3 a = div3(va, norm3(va)); /* normalize(): v / v.norm() */
    Vec3 b = div3(tdir, norm3(tdir));
    double c_alpha = dot3(a, b);
    if (c_alpha > 1.0) alpha = 0.0;
    else if (norm3(va) < 1e-6) alpha = 0.0;
    else alpha = gm_acos(c_alpha);
  }
  if (kind != 0) dynp = 0.5 * pp[PP_RHO] * norm3(va) * norm3(va);
  if (kind == 0) return alpha;
  if (kind == 1) return dynp;
  return dynp * alpha;
}
P_HD double aero_quantity(int kind, Vec3 pos, Vec3 vel, Quat q, double t, const Tables& tb) {
  double pp[PP_COLS], rp[RP_COLS];
  pos_part(pos.x, pos.y, pos.z, tb.wind, tb.n_wind, 0, pp);
  rot_part(pos.x, pos.y, pos.z, t, pp[PP_WIND_N], pp[PP_WIND_E], rp);
  return aero_quantity_col(kind, pos, vel, q, pp, rp);
}

/* ---- event-point leaves --------------------------------------------------- */
/* wrapper_coordinate.hpp:193-199 eci2geodetic -> (lat deg, lon deg, alt m) */
P_HD Vec3 eci2geodetic_deg(Vec3 pos_eci, double t) {
  double s, c;
  gm_sincos(P_OMEGA * t, &s, &c);
  Geodetic g = ecef2geodetic<3>(rot_eci2ecef(pos_eci, c, s));
  return v3(g.lat * 180.0 / P_PI, g.lon * 180.0 / P_PI, g.alt);
}

/* iip.cpp:36-150 + pybind_IIP.cpp:34-51 (fill_na = true): (lat deg, lon deg, 0) or zeros */
P_HD Vec3 iip_faa_deg(Vec3 posECEF, Vec3 velECEF) {
  const Vec3 zero = v3(0.0 * (180.0 / P_PI), 0.0 * (180.0 / P_PI), 0.0);
  double s0, c0;
  gm_sincos(P_OMEGA * 0.0, &s0, &c0);
  double r_k1 = P_RB;
  Vec3 p0 = rot_ecef2eci(posECEF, c0, s0);
  double r0 = norm3(p0);
  if (r0 < r_k1) return zero;
  Vec3 v0v = vel_ecef2eci_cs(velECEF, posECEF, c0, s0);
  double v0 = norm3(v0v);
  double eps_cos = (r0 * v0 * v0 / P_MU) - 1.0;
  if (eps_cos >= 1.0) return zero;
  double a_t = r0 / (1 - eps_cos);
  double eps_sin = dot3(p0, v0v) / gm_sqrt(P_MU * a_t);
  double eps2 = eps_cos * eps_cos + eps_sin * eps_sin;
  if (gm_sqrt(eps2) <= 1.0 && a_t * (1 - gm_sqrt(eps2)) - P_RA >= 0.0) return zero;
  double eps_k_cos = 0, eps_k_sin = 0, d_cos = 0, d_sin = 0;
  double fs, gs, Ek = 0, Fk = 0, Gk = 0, r_k2 = 0, r_k1_tmp = 0;
  for (int i = 0; i < 5; i++) {
    eps_k_cos = (a_t - r_k1) / a_t;
    if ((eps2 - eps_k_cos * eps_k_cos) < 0) return zero;
    eps_k_sin = -gm_sqrt(eps2 - eps_k_cos * eps_k_cos);
    d_cos = (eps_k_cos * eps_cos + eps_k_sin * eps_sin) / eps2;
    d_sin = (eps_k_sin * eps_cos - eps_k_cos * eps_sin) / eps2;
    fs = (d_cos - eps_cos) / (1 - eps_cos);
    gs = (d_sin + eps_sin - eps_k_sin) * gm_sqrt(a_t * a_t * a_t / P_MU);
    Ek = fs * p0.x + gs * v0v.x;
    Fk = fs * p0.y + gs * v0v.y;
    Gk = fs * p0.z + gs * v0v.z;
    r_k2 = P_RA / gm_sqrt((P_E2 / (1 - P_E2)) * (Gk / r_k1) * (Gk / r_k1) + 1);
    r_k1_tmp = r_k1;
    r_k1 = r_k2;
  }
  if (gm_fabs(r_k1_tmp - r_k2) > 1.0) return zero;
  double delta_eps = gm_atan2(d_sin, d_cos);
  double time_sec = (delta_eps + eps_sin - eps_k_sin) * gm_sqrt(a_t * a_t * a_t / P_MU);
  double phi_tmp = gm_asin(Gk / r_k2);
  double phi = gm_atan2(gm_tan(phi_tmp), 1.0 - P_E2);
  double lam = gm_atan2(Fk, Ek) - P_OMEGA * time_sec;
  return v3(phi * (180.0 / P_PI), lam * (180.0 / P_PI), 0.0);
}

/* con_waypoint.py:214-218 iip_from_eci: dimensional pos/vel, t in seconds */
P_HD Vec3 iip_from_eci_deg(Vec3 pos, Vec3 vel, double t) {
  double s, c;
  gm_sincos(P_OMEGA * t, &s, &c);
  return iip_faa_deg(rot_eci2ecef(pos, c, s), vel_eci2ecef_cs(vel, pos, c, s));
}

/* con_waypoint.py:45-51 sin_elevation; p_ant = antenna ECEF position */
P_HD double sin_elevation(Vec3 pos, double t, Vec3 p_ant) {
  double s, c;
  gm_sincos(P_OMEGA * t, &s, &c);
  Vec3 d = sub3(rot_eci2ecef(pos, c, s), p_ant);
  Vec3 dir = div3(d, norm3(d)); /* normalize(): dynamic vector v / v.norm() */
  Geodetic g = ecef2geodetic<2>(p_ant);
  Quat q_ned2ecef = quatconj(quat_ecef2ned_ll<>(g.lat, g.lon));
  Vec3 vert = quatrot(q_ned2ecef, v3(0.0, 0.0, -1.0));
  /* np.dot of two 3-vectors: BLAS ddot accumulates with fused multiply-add, ascending index
   * (the same order the kernels use for D.X; DESIGN.md H2) */
  return gm_fma(dir.z, vert.z, gm_fma(dir.y, vert.y, dir.x * vert.x));
}

/* terminal orbit (wrapper_coordinate.hpp:224-250) */
P_HD double orbit_energy(Vec3 pos, Vec3 vel) {
  double r = norm3(pos);
  double v = norm3(vel);
  return 0.5 * v * v - P_MU / r;
}
P_HD double angular_momentum(Vec3 pos, Vec3 vel) { return norm3(cross3(pos, vel)); }
P_HD double inclination_rad(Vec3 pos, Vec3 vel) {
  Vec3 h = cross3(pos, vel);
  return gm_acos(h.z / norm3(h));
}

/* Coordinate.cpp:197-245 orbital_elements, only a and e (what the shipped
 * user constraint reads: example/user_constraints.py:133-137) */
P_HD void orbital_a_e(Vec3 pos, Vec3 vel, double* a_out, double* e_out) {
  Vec3 nr = normalized3(pos);
  Vec3 c = cross3(pos, vel);
  Vec3 f = sub3(cross3(vel, c), scale3(P_MU, nr));
  double p = dot3(c, c) / P_MU;
  double e = norm3(f) / P_MU;
  *a_out = p / (1.0 - e * e);
  *e_out = e;
}

/* Coordinate.cpp:197-245 orbital_elements: a, e, inclination, ascending node, argument of perigee, true anomaly (radians) */
P_HD void orbital_elements6(Vec3 pos, Vec3 vel, double* out) {
  const Vec3 nr = normalized3(pos);
  const Vec3 c = cross3(pos, vel);
  const Vec3 f = sub3(cross3(vel, c), scale3(P_MU, nr));
  const Vec3 c1 = normalized3(c);
  const Vec3 f1 = normalized3(f);
  const double inc = gm_acos(c1.z);
  double asc = 0.0, argp = 0.0;
  if (inc > 1.0e-10) {
    asc = gm_atan2(c1.x, -c1.y);
    double sa, ca;
    gm_sincos(asc, &sa, &ca);
    argp = gm_acos(dot3(v3(ca, sa, 0.0), f1));
    if (f.z < 0.0) argp *= -1.0;
  } else {
    if (norm3(f) > 1.0e-10) argp = gm_atan2(f.y, f.x);
  }
  const double p = dot3(c, c) / P_MU;
  const double e = norm3(f) / P_MU;
  double ta = gm_acos(dot3(f1, nr));
  if (dot3(vel, pos) < 0.0) ta = 2.0 * P_PI - ta;
  if (asc < 0.0) asc += 2.0 * P_PI;
  if (argp < 0.0) argp += 2.0 * P_PI;
  if (ta < 0.0) ta += 2.0 * P_PI;
  out[0] = p / (1.0 - e * e); out[1] = e; out[2] = inc; out[3] = asc; out[4] = argp; out[5] = ta;
}

/* one orbit quantity of a user built-in (include/gelato_b200.h: GEQ_*), from the elements / leaves the reference's
 * own user constraints would call (example/user_constraints.py:96-139) */
P_HD double orbit_quantity(int code, Vec3 pos, Vec3 vel) {
  if (code == 5) return orbit_energy(pos, vel);
  if (code == 6) return angular_momentum(pos, vel);
  double el[6];
  orbital_elements6(pos, vel, el);
  switch (code) {
    case 0: return el[0] * (1.0 - el[1]);
    case 1: return el[0] * (1.0 + el[1]);
    case 2: return el[0];
    case 3: return el[1];
    default: return el[2] * 180.0 / P_PI; /* the wrapper returns degrees: wrapper_coordinate.hpp:204 */
  }
}

#endif /* GELATO_B200_PHYSICS_H_ */
