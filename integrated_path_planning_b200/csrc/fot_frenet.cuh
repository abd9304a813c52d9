// fot_frenet.cuh -- nearest point on the reference path for a batch of ego positions (cc.py:202-283, the search of
// find_nearest_point_on_path with the `_prev_s` window cache), as frenet_host.BatchCoordinateConverter.nearest_s
// restates it.  One warp per query.
//
// The answer has to be the host's bit for bit, but the host's spline positions use NumPy's array `dx ** 3.0`, whose
// last bit is the host CPU's pow and not something the device can reproduce.  So (DESIGN.md section 4e):
//   * every other operation of the search is the host's operation (compiled with -fmad=false; dx2 = dx * dx is what
//     NumPy's `** 2.0` computes; linspace is `k * step + lo`, last sample `hi`; max / min / step * 0.5 are plain);
//   * a position is evaluated twice, with the cube moved kCubeUlps ulps down and up.  Rounded add and multiply are
//     monotone, so every cube in between -- the host's included, if it lies within kCubeUlps ulps of dx * dx * dx --
//     gives a position between the two results.  Equal results pin the host's position exactly; otherwise the
//     position is carried as that interval;
//   * a decision `a < b` between two distances is taken only when it is certain: the bounds are further apart than
//     kNear relative (the host's np.hypot / math.hypot and the device's hypot are each within a few ulps of the
//     exact distance of the same point), or both candidates are the same arc length (identical on both sides);
//   * a query with any decision that is not certain, or any unusual input (NaN, inf, an empty window), gets
//     status 1 and the host recomputes it.
#pragma once
#include "fot_device.cuh"

namespace fot {

constexpr int kCubeUlps = 4;                                   // host dx ** 3.0 assumed within 4 ulps of dx * dx * dx
constexpr double kNear = 16.0 * 2.220446049250313e-16;         // BatchCoordinateConverter.NEAR
constexpr double kWindow = 10.0;                               // CoordinateConverter.WINDOW
constexpr int kWindowSamples = 100;                            // CoordinateConverter.WINDOW_SAMPLES
constexpr double kGlobalStep = 0.1;                            // CoordinateConverter.GLOBAL_STEP

// dx * dx * dx, the device's cube (NumPy's `dx ** 2.0` is dx * dx, then one more product).
__device__ __forceinline__ double near_cube(double dx) { return dx * dx * dx; }

// Interval of a distance: lo <= the host's value <= hi, up to the hypot error that kNear covers.
struct NearDist {
  double lo, hi;
};

// Bounds of |x - p| for p in [p0, p1] (p0 <= p1): rounded subtraction is monotone in p.
__device__ __forceinline__ void near_abs_bounds(double x, double p0, double p1, double& a_lo, double& a_hi) {
  const double e_lo = x - p1, e_hi = x - p0;
  if (e_lo >= 0.0) { a_lo = e_lo; a_hi = e_hi; }
  else if (e_hi <= 0.0) { a_lo = -e_hi; a_hi = -e_lo; }
  else { a_lo = 0.0; a_hi = fmax(-e_lo, e_hi); }
}

// Distance from (x, y) to the path point at arc length s, as an interval over every cube within kCubeUlps ulps of
// the device's.  NaN outside the knots (cs.py:62), which makes every decision about it uncertain.
__device__ __forceinline__ NearDist near_dist(const Plan& P, double s, double x, double y) {
  const int nx = P.cfg.nx;
  if (!(s >= P.knots[0] && s <= P.knots[nx - 1])) return NearDist{qnan(), qnan()};
  int lo = 0, hi = nx;                                 // searchsorted(side='right') - 1, clipped (cs.py:162-165)
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (P.knots[mid] <= s) lo = mid + 1; else hi = mid;
  }
  int seg = lo - 1;
  seg = seg < 0 ? 0 : (seg > nx - 2 ? nx - 2 : seg);
  const double dx = s - P.knots[seg];
  const double dx2 = dx * dx;
  double c0 = near_cube(dx), c1 = c0;
#pragma unroll
  for (int k = 0; k < kCubeUlps; ++k) { c0 = nextafter(c0, -HUGE_VAL); c1 = nextafter(c1, HUGE_VAL); }
  const double xs = P.xa[seg] + P.xb[seg] * dx + P.xc[seg] * dx2;     // cs.py:73-74, left to right
  const double ys = P.ya[seg] + P.yb[seg] * dx + P.yc[seg] * dx2;
  const double xd = P.xd[seg], yd = P.yd[seg];
  const double px0 = xs + xd * c0, px1 = xs + xd * c1;
  const double py0 = ys + yd * c0, py1 = ys + yd * c1;
  double ax_lo, ax_hi, ay_lo, ay_hi;
  near_abs_bounds(x, fmin(px0, px1), fmax(px0, px1), ax_lo, ax_hi);
  near_abs_bounds(y, fmin(py0, py1), fmax(py0, py1), ay_lo, ay_hi);
  NearDist g;
  g.lo = hypot(ax_lo, ay_lo);
  g.hi = ax_lo == ax_hi && ay_lo == ay_hi ? g.lo : hypot(ax_hi, ay_hi);
  if (px0 != px0 || py0 != py0 || px1 != px1 || py1 != py1) g.lo = g.hi = qnan();
  return g;
}

// The host's `g_a < g_b`: 1 certainly true, -1 certainly false, 0 not certain (NaN included).
__device__ __forceinline__ int near_less(const NearDist& a, double s_a, const NearDist& b, double s_b) {
  if (s_a == s_b) return -1;                           // same point on both sides: equal distances
  if (b.lo - a.hi > kNear * fmax(a.hi, b.lo)) return 1;
  if (a.lo - b.hi > kNear * fmax(b.hi, a.lo)) return -1;
  return 0;
}

// Three-valued `p and q`.
__device__ __forceinline__ int near_and(int p, int q) { return (p < 0 || q < 0) ? -1 : (p > 0 && q > 0 ? 1 : 0); }

// First minimum of the distance over the samples k * step + lo (k < n - 1) and hi (k = n - 1) -- np.linspace's
// arithmetic -- across the lanes of the warp.  Returns the chosen sample's arc length; `sure` false unless every
// other sample is certainly farther (the runner-up's lower bound against the winner's upper bound).
__device__ __forceinline__ double near_argmin(const Plan& P, double x, double y, double lo, double hi, double step, int n,
                                              bool& sure) {
  const int lane = threadIdx.x & 31;
  double b_lo = INFINITY, b_hi = INFINITY, r_lo = INFINITY;   // best (lower, upper bound), runner-up lower bound
  int b_k = 0x7fffffff;
  bool nan = false;
  for (int k = lane; k < n; k += 32) {
    const double s = k == n - 1 ? hi : (double)k * step + lo;
    const NearDist g = near_dist(P, s, x, y);
    nan |= !(g.lo == g.lo);
    if (g.lo < b_lo) { r_lo = b_lo; b_lo = g.lo; b_hi = g.hi; b_k = k; }
    else r_lo = fmin(r_lo, g.lo);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const double o_lo = __shfl_xor_sync(0xffffffffu, b_lo, off), o_hi = __shfl_xor_sync(0xffffffffu, b_hi, off);
    const double o_r = __shfl_xor_sync(0xffffffffu, r_lo, off);
    const int o_k = __shfl_xor_sync(0xffffffffu, b_k, off);
    if (o_lo < b_lo || (o_lo == b_lo && o_k < b_k)) {
      r_lo = fmin(o_r, b_lo);
      b_lo = o_lo; b_hi = o_hi; b_k = o_k;
    } else {
      r_lo = fmin(r_lo, o_lo);
    }
  }
  nan = __any_sync(0xffffffffu, nan);
  sure = !nan && b_k < n && r_lo - b_hi > kNear * fmax(b_hi, r_lo);
  return b_k == n - 1 ? hi : (double)b_k * step + lo;
}

// One warp per query.  x, y, prev_s (NaN: no cache) [n]; s_out, status [n].  prev_s is read, never written.  kRoutes:
// point q is searched on its own route (R; a bad route id gives status 1).  A template parameter, so that the
// unrouted kernel keeps its code and registers.
template <bool kRoutes>
__device__ __forceinline__ void nearest_s_body(const Plan& P_, const Routes& R, int n, const double* __restrict__ xs,
                                               const double* __restrict__ ys, const double* __restrict__ prev_s,
                                               double* __restrict__ s_out, int32_t* __restrict__ status) {
  const int q = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (q >= n) return;                                  // whole warps leave together
  Plan PR_;
  if constexpr (kRoutes) {
    if (!route_plan(P_, R, q, PR_)) {
      if (lane == 0) { s_out[q] = qnan(); status[q] = 1; }
      return;
    }
  }
  const Plan& P = kRoutes ? PR_ : P_;
  const double x = xs[q], y = ys[q], prev = prev_s[q];
  const double end = P.knots[P.cfg.nx - 1];            // reference_path.s[-1]
  bool sure = isfinite(x) && isfinite(y) && (isfinite(prev) || isnan(prev)) && end > 0.0;
  double best = 0.0;
  if (sure) {
    bool global = true;
    if (!isnan(prev)) {                                // cached window (cc.py:221-248)
      const double a = prev - kWindow, b = prev + kWindow;
      const double lo = a > 0.0 ? a : 0.0;             // max(0.0, prev - W)
      const double hi = b < end ? b : end;             // min(path_end, prev + W)
      const double step = (hi - lo) / (double)(kWindowSamples - 1);
      if (step > 0.0) {                                // step == 0: np.linspace's other branch, left to the host
        best = near_argmin(P, x, y, lo, hi, step, kWindowSamples, sure);
        global = (fabs(best - lo) < 1e-3 && lo > 0.0) || (fabs(best - hi) < 1e-3 && hi < end);
      } else {
        sure = false;
      }
    }
    if (sure && global) {                              // np.linspace(0, end, n) (cc.py:319-339)
      const double ng = end / kGlobalStep;
      const int n_g = ng < 100.0 ? 100 : (ng >= 2.0e9 ? -1 : (int)ng);
      if (n_g < 0) sure = false;
      else best = near_argmin(P, x, y, 0.0, end, end / (double)(n_g - 1), n_g, sure);
    }
  }
  // 20 three-point refinements (cc.py:253-280): lanes 0, 1, 2 evaluate s_lo, s_hi, best
  double step = 0.2;
  for (int it = 0; it < 20 && sure; ++it) {
    const double a = best - step, b = best + step;
    const double s_lo = a > 0.0 ? a : 0.0;            // max(0, best - step)
    const double s_hi = b < end ? b : end;            // min(path_end, best + step)
    NearDist g{0.0, 0.0};
    if (lane < 3) g = near_dist(P, lane == 0 ? s_lo : (lane == 1 ? s_hi : best), x, y);
    const NearDist g_lo{__shfl_sync(0xffffffffu, g.lo, 0), __shfl_sync(0xffffffffu, g.hi, 0)};
    const NearDist g_hi{__shfl_sync(0xffffffffu, g.lo, 1), __shfl_sync(0xffffffffu, g.hi, 1)};
    const NearDist g_c{__shfl_sync(0xffffffffu, g.lo, 2), __shfl_sync(0xffffffffu, g.hi, 2)};
    const int go_lo = near_and(near_less(g_lo, s_lo, g_c, best), near_less(g_lo, s_lo, g_hi, s_hi));
    if (go_lo > 0) { best = s_lo; continue; }
    const int go_hi = near_and(near_less(g_hi, s_hi, g_c, best), near_less(g_hi, s_hi, g_lo, s_lo));
    if (go_lo == 0 || go_hi == 0) { sure = false; break; }
    if (go_hi > 0) best = s_hi;
    else step = step * 0.5;
  }
  if (lane == 0) {
    s_out[q] = sure ? best : qnan();
    status[q] = sure ? 0 : 1;
  }
}
__global__ void __launch_bounds__(256) fot_nearest_s(const Plan P, int n, const double* __restrict__ xs,
                                                     const double* __restrict__ ys, const double* __restrict__ prev_s,
                                                     double* __restrict__ s_out, int32_t* __restrict__ status) {
  nearest_s_body<false>(P, Routes{}, n, xs, ys, prev_s, s_out, status);
}
__global__ void __launch_bounds__(256) fot_nearest_s_routed(const Plan P, const Routes R, int n, const double* __restrict__ xs,
                                                            const double* __restrict__ ys, const double* __restrict__ prev_s,
                                                            double* __restrict__ s_out, int32_t* __restrict__ status) {
  nearest_s_body<true>(P, R, n, xs, ys, prev_s, s_out, status);
}

}  // namespace fot
