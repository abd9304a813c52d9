// fot_device.cuh -- device-side numerics of the Frenet candidate sweep (sm_100a).
//
// Compiled with -fmad=false: every expression below keeps the reference's NumPy
// association order and rounding (one rounding per * and +); fused multiply-adds
// appear only where written explicitly as fma().  Reference citations are to
// /root/reference/src/planning/frenet_planner.py ("fp.py"),
// src/planning/cubic_spline.py ("cs.py") and src/core/coordinate_converter.py ("cc.py").
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include "fot.h"

namespace fot {

// Planner constants resident on the device (pointers into one device blob).
struct Plan {
  fot_config_t cfg;
  const double *T, *inv4, *inv5, *Tb, *inv4b, *inv5b, *d_grid;
  const int32_t *n_steps, *n_steps_b;
  const double *knots, *xa, *xb, *xc, *xd, *ya, *yb, *yc, *yd;
  int32_t n_t_max;
  int32_t d_sorted;        // d_grid is non-decreasing (the reference's grid always is)
  double d_min, d_max;     // extreme lateral targets
};

// Per-query reference paths (fot_add_route / fot_set_routes; DESIGN.md section 4h).  All null: every query plans on the
// Plan's own path.  Route r's nine spline tables lie at tab + off[r], each nx[1 + r] doubles long (knots | x: a b c d |
// y: a b c d; the b and d tables use nx - 1 of them); nx[0] is the number of routes.  Route 0 is the Plan's path.
struct Routes {
  const int32_t* id;     // [n_q] route of query q (already offset to the launch's first query)
  const int32_t* nx;     // [1 + n_routes]
  const int32_t* off;    // [n_routes]
  const double* tab;
};

// One batch, device pointers.
struct Batch {
  int32_t n_q, n_v_max;
  const double *frenet, *target, *limits, *stop_dist, *v_grid;
  const int32_t* n_v;
  int32_t n_static, static_per_query;
  int32_t S, P, T_obs, dyn_mode;
  // the sweep kernels read the caller's tensors directly:
  const double* dyn_raw;      // [n_q][S][P][T_obs][2] (reference layout) or null
  const double* static_raw;   // [n_q or 1][M][2] or null
  const float4* dyn_box;      // [n_q][S*P] trajectory boxes (xmin, xmax, ymin, ymax) from fot_aabb_prepass
  const double* cost_tab;     // [n_q][n_T*(n_v_max + 2 n_d) + 3 n_B] jerk sums / terminal offsets from fot_cost_prepass
  // Per-query routes, null unless the handle has a route binding.  These 32 bytes were padding before routes existed and
  // are kept in any case: Out and the geometry follow Batch in the sweep kernels' parameters, and without them ptxas
  // schedules fot_sweep_pairs differently -- the sweep of bench.py ran 1.2 % slower (1.597 against 1.578 ms; B200, 1000 W).
  Routes rt;
};

// V = P with the spline tables and knot count of query q's route.  Without routes V is P.  False for a route id outside
// [0, n_routes): that query plans nothing, and no table is read for it.
__device__ __forceinline__ bool route_plan(const Plan& P, const Routes& R, int q, Plan& V) {
  V = P;
  if (!R.id) return true;
  const int r = R.id[q];
  if (r < 0 || r >= R.nx[0]) return false;
  const int nx = R.nx[1 + r];
  const double* t = R.tab + R.off[r];
  V.cfg.nx = nx;
  V.knots = t;
  V.xa = t + nx;     V.xb = t + 2 * nx; V.xc = t + 3 * nx; V.xd = t + 4 * nx;
  V.ya = t + 5 * nx; V.yb = t + 6 * nx; V.yc = t + 7 * nx; V.yd = t + 8 * nx;
  return true;
}

struct Out {
  int32_t* best_idx; double* best_cost; int32_t* stats; int32_t* winner_len; double* winner;
  uint8_t* cand_cat; double* cand_cost; int32_t cand_stride;
  double* part_cost; int32_t* part_idx;   // [n_q][blocks_per_query] partial arg-min
  // Mirror of the winner block (fot_set_result_mirror): a second set of result arrays -- typically PEER memory on the
  // gather root of a multi-GPU job, mapped over NVLink -- that fot_winner writes together with the local ones.  All null: none.
  int32_t* m_best_idx; double* m_best_cost; int32_t* m_stats; int32_t* m_winner_len; double* m_winner;
};

__device__ __forceinline__ double qnan() { return __longlong_as_double(0x7ff8000000000000LL); }

// ---- coefficient solve: `b @ A_inv.T` (fp.py:640, :683) -------------------------------
// NumPy hands this product to BLAS; on the x86-64 builds in this image the accumulation
// is a left-to-right FMA chain for >= 2 rows and (k = 1, 0, 2) for a single row (brake
// candidates, target_speed = 0).  `single` selects the latter.
__device__ __forceinline__ void apply_inv2(const double* __restrict__ A, double r0, double r1,
                                           bool single, double& o0, double& o1) {
  if (!single) {
    o0 = fma(r1, A[1], r0 * A[0]);
    o1 = fma(r1, A[3], r0 * A[2]);
  } else {
    o0 = fma(r0, A[0], r1 * A[1]);
    o1 = fma(r0, A[2], r1 * A[3]);
  }
}
__device__ __forceinline__ void apply_inv3(const double* __restrict__ A, double r0, double r1, double r2,
                                           bool single, double& o0, double& o1, double& o2) {
  if (!single) {
    o0 = fma(r2, A[2], fma(r1, A[1], r0 * A[0]));
    o1 = fma(r2, A[5], fma(r1, A[4], r0 * A[3]));
    o2 = fma(r2, A[8], fma(r1, A[7], r0 * A[6]));
  } else {
    o0 = fma(r2, A[2], fma(r0, A[0], r1 * A[1]));
    o1 = fma(r2, A[5], fma(r0, A[3], r1 * A[4]));
    o2 = fma(r2, A[8], fma(r0, A[6], r1 * A[7]));
  }
}

// Quartic longitudinal profile (fp.py:619-647).  `hold`: last polynomial sample; beyond it the
// brake-ladder padding applies (position held, derivatives zero; fp.py:487-499).
struct Lon {
  double a0, a1, a2, a3, a4;
  int hold;
};
__device__ __forceinline__ Lon lon_solve(const double* __restrict__ fs, double tv, double T,
                                         const double* __restrict__ inv4, bool single, int hold) {
  Lon L;
  L.a0 = fs[0];
  L.a1 = fs[1];
  L.a2 = fs[2] / 2.0;
  const double r0 = tv - L.a1 - 2.0 * L.a2 * T;
  const double r1 = -2.0 * L.a2;
  apply_inv2(inv4, r0, r1, single, L.a3, L.a4);
  L.hold = hold;
  return L;
}
// tt = shared table [NT][kTT] of t, t^2, t^3, t^4, t^5 (one row per sample) built as fp.py:594-598.
constexpr int kTT = 6;
__device__ __forceinline__ void tt_fill(double* tt, int n, double dt) {
  const double t = (double)n * dt;
  const double t2 = t * t, t3 = t2 * t, t4 = t2 * t2, t5 = t4 * t;
  double* r = tt + kTT * n;
  r[0] = t; r[1] = t2; r[2] = t3; r[3] = t4; r[4] = t5; r[5] = 0.0;
}
__device__ __forceinline__ double lon_p0(const Lon& L, const double* tt, int n) {
  const double* r = tt + kTT * (n > L.hold ? L.hold : n);
  return L.a0 + L.a1 * r[0] + L.a2 * r[1] + L.a3 * r[2] + L.a4 * r[3];
}
__device__ __forceinline__ double lon_p1(const Lon& L, const double* tt, int n) {
  if (n > L.hold) return 0.0;
  const double* r = tt + kTT * n;
  return L.a1 + 2.0 * L.a2 * r[0] + 3.0 * L.a3 * r[1] + 4.0 * L.a4 * r[2];
}
__device__ __forceinline__ double lon_p2(const Lon& L, const double* tt, int n) {
  if (n > L.hold) return 0.0;
  const double* r = tt + kTT * n;
  return 2.0 * L.a2 + 6.0 * L.a3 * r[0] + 12.0 * L.a4 * r[1];
}
__device__ __forceinline__ double lon_p3(const Lon& L, const double* tt, int n) {
  if (n > L.hold) return 0.0;
  return 6.0 * L.a3 + 24.0 * L.a4 * tt[kTT * n];
}

// Quintic lateral profile (fp.py:660-691).
struct Lat {
  double a0, a1, a2, a3, a4, a5;
  int hold;
};
__device__ __forceinline__ Lat lat_solve(const double* __restrict__ fs, double di, double T,
                                         const double* __restrict__ inv5, bool single, int hold) {
  Lat L;
  L.a0 = fs[3];
  L.a1 = fs[4];
  L.a2 = fs[5] / 2.0;
  const double r0 = di - L.a0 - L.a1 * T - L.a2 * T * T;
  const double r1 = -L.a1 - 2.0 * L.a2 * T;
  const double r2 = -2.0 * L.a2;
  apply_inv3(inv5, r0, r1, r2, single, L.a3, L.a4, L.a5);
  L.hold = hold;
  return L;
}
__device__ __forceinline__ double lat_p0(const Lat& L, const double* tt, int n) {
  const double* r = tt + kTT * (n > L.hold ? L.hold : n);
  return L.a0 + L.a1 * r[0] + L.a2 * r[1] + L.a3 * r[2] + L.a4 * r[3] + L.a5 * r[4];
}
__device__ __forceinline__ double lat_p1(const Lat& L, const double* tt, int n) {
  if (n > L.hold) return 0.0;
  const double* r = tt + kTT * n;
  return L.a1 + 2.0 * L.a2 * r[0] + 3.0 * L.a3 * r[1] + 4.0 * L.a4 * r[2] + 5.0 * L.a5 * r[3];
}
__device__ __forceinline__ double lat_p2(const Lat& L, const double* tt, int n) {
  if (n > L.hold) return 0.0;
  const double* r = tt + kTT * n;
  return 2.0 * L.a2 + 6.0 * L.a3 * r[0] + 12.0 * L.a4 * r[1] + 20.0 * L.a5 * r[2];
}
__device__ __forceinline__ double lat_p3(const Lat& L, const double* tt, int n) {
  if (n > L.hold) return 0.0;
  const double* r = tt + kTT * n;
  return 6.0 * L.a3 + 24.0 * L.a4 * r[0] + 60.0 * L.a5 * r[1];
}

// Lateral offset and its first two time derivatives at time t by Horner's scheme with running
// derivatives (12 FMAs, needs only t).  Used by the sweep's validity and collision passes; differs from
// the reference-order lat_p0/1/2 by a few ulp.  The cost and the returned winner use the latter.
__device__ __forceinline__ void lat_fast(const Lat& L, double t, double& d, double& d1, double& d2) {
  double p = fma(L.a5, t, L.a4), dp = L.a5, ddp;
  ddp = dp;             dp = fma(dp, t, p);  p = fma(p, t, L.a3);
  ddp = fma(ddp, t, dp); dp = fma(dp, t, p);  p = fma(p, t, L.a2);
  ddp = fma(ddp, t, dp); dp = fma(dp, t, p);  p = fma(p, t, L.a1);
  ddp = fma(ddp, t, dp); dp = fma(dp, t, p);  p = fma(p, t, L.a0);
  d = p; d1 = dp; d2 = 2.0 * ddp;
}
__device__ __forceinline__ double lat_fast0(const Lat& L, double t) {
  return fma(fma(fma(fma(fma(L.a5, t, L.a4), t, L.a3), t, L.a2), t, L.a1), t, L.a0);
}

// np.sum over a contiguous float64 vector: NumPy's pairwise summation (8 interleaved
// accumulators per <=128-element block, halving above that).  The jerk costs fp.py:718,:722
// go through it, so the cost -- and with it the arg-min -- only reproduces with this order.
// np_block_sum is one block; np_pairwise_sum_flat is the whole sum for any n.
template <class F>
__device__ __forceinline__ double np_block_sum(const F& f, int lo, int n) {   // n <= 128
  if (n < 8) {
    double r = 0.0;
    for (int i = 0; i < n; ++i) r += f(lo + i);
    return r;
  }
  double r0 = f(lo), r1 = f(lo + 1), r2 = f(lo + 2), r3 = f(lo + 3);
  double r4 = f(lo + 4), r5 = f(lo + 5), r6 = f(lo + 6), r7 = f(lo + 7);
  int i = 8;
  const int stop = n - (n % 8);
  for (; i < stop; i += 8) {
    r0 += f(lo + i);     r1 += f(lo + i + 1); r2 += f(lo + i + 2); r3 += f(lo + i + 3);
    r4 += f(lo + i + 4); r5 += f(lo + i + 5); r6 += f(lo + i + 6); r7 += f(lo + i + 7);
  }
  double res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
  for (; i < n; ++i) res += f(lo + i);
  return res;
}
// Above 128 elements NumPy halves the range (the left half rounded down to a multiple of 8) and adds the two halves'
// sums.  That split tree is walked here with an explicit stack rather than by recursion: a recursive form takes a
// 200-byte stack frame per level, and sums of a few thousand terms overflow the default 1 KB thread stack.
template <class F>
__device__ double np_pairwise_sum_flat(const F& f, int n) {
  if (n <= 128) return np_block_sum(f, 0, n);
  int s_lo[32], s_n[32], s_state[32];                   // depth <= log2(n / 128) + 1 < 32
  double s_left[32];
  int sp = 0;
  s_lo[0] = 0; s_n[0] = n; s_state[0] = 0;
  double ret = 0.0;
  for (;;) {
    const int lo = s_lo[sp], m = s_n[sp];
    int m2 = m / 2;
    m2 -= m2 % 8;
    if (m <= 128) {
      ret = np_block_sum(f, lo, m);
      --sp;
    } else if (s_state[sp] == 0) {                      // descend left
      s_state[sp] = 1;
      ++sp; s_lo[sp] = lo; s_n[sp] = m2; s_state[sp] = 0;
      continue;
    } else if (s_state[sp] == 1) {                      // left done: descend right
      s_left[sp] = ret; s_state[sp] = 2;
      ++sp; s_lo[sp] = lo + m2; s_n[sp] = m - m2; s_state[sp] = 0;
      continue;
    } else {                                            // both done: left + right
      ret = s_left[sp] + ret;
      --sp;
    }
    if (sp < 0) return ret;
  }
}

// Reference-line sample at arc length s (cs.py:47-166, :215-288).  NaN outside the knot range.
struct RefPt {
  double rx, ry, rth, rk, rdk;
};
__device__ __forceinline__ RefPt spline_ref(const Plan& P, double s) {
  RefPt o;
  const int nx = P.cfg.nx;
  if (!(s >= P.knots[0] && s <= P.knots[nx - 1])) {   // cs.py:62 (inclusive; NaN s fails both)
    o.rx = o.ry = o.rth = o.rk = o.rdk = qnan();
    return o;
  }
  int lo = 0, hi = nx;                                 // searchsorted(side='right') (cs.py:162)
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (P.knots[mid] <= s) lo = mid + 1; else hi = mid;
  }
  int seg = lo - 1;
  seg = seg < 0 ? 0 : (seg > nx - 2 ? nx - 2 : seg);   // cs.py:165
  const double dx = s - P.knots[seg];
  const double dx2 = dx * dx;
  const double dx3 = dx2 * dx;
  const double xa = P.xa[seg], xb = P.xb[seg], xc = P.xc[seg], xd = P.xd[seg];
  const double ya = P.ya[seg], yb = P.yb[seg], yc = P.yc[seg], yd = P.yd[seg];
  o.rx = xa + xb * dx + xc * dx2 + xd * dx3;           // cs.py:73-74
  o.ry = ya + yb * dx + yc * dx2 + yd * dx3;
  const double x1 = xb + 2.0 * xc * dx + 3.0 * xd * dx2;   // cs.py:100
  const double y1 = yb + 2.0 * yc * dx + 3.0 * yd * dx2;
  const double x2 = 2.0 * xc + 6.0 * xd * dx;              // cs.py:125
  const double y2 = 2.0 * yc + 6.0 * yd * dx;
  const double x3 = 6.0 * xd, y3 = 6.0 * yd;               // cs.py:149
  o.rth = atan2(y1, x1);                                   // cs.py:287
  const double D = x1 * x1 + y1 * y1;
  const double rD = sqrt(D);
  const double D15 = D * rD;                               // D ** 1.5
  const double D25 = D * D * rD;                           // D ** 2.5
  o.rk = (y2 * x1 - x2 * y1) / D15;                        // cs.py:246
  const double a = x1 * y2 - y1 * x2;
  const double b = x1 * y3 - y1 * x3;
  const double c = x1 * x2 + y1 * y2;
  o.rdk = b / D15 - 3.0 * a * c / D25;                     // cs.py:273
  return o;
}

// Frenet -> Cartesian at one sample (fp.py:792-799 then cc.py:128-158).
struct CartPt {
  double x, y, kappa, v, a, ang;   // ang = delta_theta + rtheta, yaw = wrap(ang)
};
__device__ __forceinline__ CartPt to_cartesian(double rx, double ry, double cth, double sth, double rth,
                                               double rk, double rdk, double sd, double sdd,
                                               double d, double dd_t, double ddd_t) {
  CartPt c;
  double d_p = 0.0, d_pp = 0.0;
  if (fabs(sd) > 1e-3) {                                   // fp.py:792 EPS_S_DOT
    d_p = dd_t / sd;
    d_pp = (ddd_t - d_p * sdd) / (sd * sd);
  }
  c.x = rx - sth * d;
  c.y = ry + cth * d;
  const double q = 1.0 - rk * d;
  const double tan_d = d_p / q;
  const double dth = atan2(d_p, q);
  const double cos_d = cos(dth);
  c.ang = dth + rth;
  const double m = rdk * d + rk * d_p;
  c.kappa = (((d_pp + m * tan_d) * cos_d * cos_d) / q + rk) * cos_d / q;
  const double d_dot = d_p * sd;
  c.v = sqrt(q * q * sd * sd + d_dot * d_dot);
  const double dth_p = q / cos_d * c.kappa - rk;
  c.a = sdd * q / cos_d + sd * sd / cos_d * (d_p * dth_p - m);
  return c;
}
// Same conversion for the sweep's validity chain, with the transcendentals removed:
//   cos(atan2(d', q)) = q / hypot(q, d'),  v = |s_dot| * hypot(q, d'),  divisions by s_dot, q and
//   cos(delta) replaced by multiplication with one reciprocal each.
// Values differ from to_cartesian() by a few ulp (<= 1e-14 relative), far inside the 1e-9 parity
// bound; the winner's returned sequences are regenerated with the reference-order to_cartesian().
// inv_sd / inv_sd2 = 1/s_dot and its square, or 0 when |s_dot| <= EPS_S_DOT (fp.py:792-799).
struct KinPt {
  double kappa, v, a, d_p, q;
};
__device__ __forceinline__ KinPt kinematics_fast(double rk, double rdk, double sd, double sdd, double inv_sd,
                                                 double inv_sd2, double d, double dd_t, double ddd_t) {
  KinPt c;
  c.d_p = dd_t * inv_sd;
  const double d_pp = (ddd_t - c.d_p * sdd) * inv_sd2;
  c.q = 1.0 - rk * d;
  const double h2 = fma(c.q, c.q, c.d_p * c.d_p);
  const double rh = rsqrt(h2);
  const double h = h2 * rh;
  const double rq = 1.0 / c.q;
  const double cos_d = c.q * rh;
  const double tan_d = c.d_p * rq;
  const double m = fma(rdk, d, rk * c.d_p);
  const double cq = cos_d * rq;
  c.kappa = fma(fma(m, tan_d, d_pp) * cos_d, cq, rk) * cq;
  c.v = fabs(sd) * h;
  const double rc = h * rq;                       // 1 / cos(delta)
  const double dth_p = fma(c.q * rc, c.kappa, -rk);
  c.a = fma(sdd * c.q, rc, sd * sd * rc * fma(c.d_p, dth_p, -m));
  return c;
}

// normalize_angle (cc.py:173-182): np.angle(np.exp(1j*a)) = atan2(sin a, cos a).
__device__ __forceinline__ double wrap_angle(double a) {
  double s, c;
  sincos(a, &s, &c);
  return atan2(s, c);
}

// Lexicographic (cost, index) minimum: first strict minimum in generation order (fp.py:1254-1257).  A NaN value never
// replaces the running minimum.  I: int for candidate indices, long long for the flat indices of fot_assess.
template <class I>
__device__ __forceinline__ void argmin_merge(double& c, I& i, double oc, I oi) {
  if (oc < c || (oc == c && oi < i)) { c = oc; i = oi; }
}

// Centre of one footprint circle: the path point moved `off` along the heading (hx, hy) = (cos yaw, sin yaw)
// (footprint.py:44-45, fp.py:1152-1160).
__device__ __forceinline__ double2 footprint_centre(double x, double y, double hx, double hy, double off) {
  return make_double2(x + off * hx, y + off * hy);
}

// 1/x and 1/sqrt(x) to fp64 accuracy from the fp32 MUFU seed and two Newton steps (branch-free; the
// library versions carry slow paths for denormals and cost three times as many instructions).  Used for
// quantities that only feed the validity chain (a few ulp are immaterial there); arguments are O(1).
__device__ __forceinline__ double rcp_nr(double a) {
  double x = (double)__frcp_rn((float)a);
  x = fma(x, fma(-a, x, 1.0), x);
  x = fma(x, fma(-a, x, 1.0), x);
  return x;
}
__device__ __forceinline__ double rsqrt_nr(double a) {
  double y = (double)rsqrtf((float)a);
  const double h = 0.5 * a;
  y = fma(y, fma(-h * y, y, 0.5), y);
  y = fma(y, fma(-h * y, y, 0.5), y);
  return y;
}

// Time powers of one sample, built as the reference's TimeCache does (fp.py:594-598).
struct TPow {
  double t, t2, t3, t4, t5;
};
__device__ __forceinline__ TPow tpow(int n, double dt) {
  TPow r;
  r.t = (double)n * dt;
  r.t2 = r.t * r.t; r.t3 = r.t2 * r.t; r.t4 = r.t2 * r.t2; r.t5 = r.t4 * r.t;
  return r;
}

// Order-preserving float <-> unsigned map for atomicMin / atomicMax on floats.
__device__ __forceinline__ unsigned f2ord(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

}  // namespace fot
