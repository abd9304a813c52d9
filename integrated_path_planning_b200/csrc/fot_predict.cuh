// fot_predict.cuh -- the predictor's post-processing on the device (SURVEY.md section 8f, rank 1):
// everything between "raw predictor output / last two observations" and the obstacle tensor
// [n_q][S][P][T_obs][2] that the sweep reads, so that batched roll-outs never upload that tensor.
//
//   fot_cv_kernel        TrajectoryPredictor.predict_cv          (trajectory_predictor.py:188-231)
//   fot_resample_kernel  TrajectoryPredictor.process_prediction  (:233-313): np.interp onto the planner
//                        grid, the constant-fill rule, the clamped tail extrapolation
//   fot_best_sample_*    closest-to-mean sample of predict_single_best (:343-351)
//   all three            the t = 0 prepend of IntegratedSimulator._update_prediction
//                        (integrated_simulator.py:503-525), including its "already has the current
//                        positions" exception
// Arithmetic follows the reference operation by operation (the file is compiled with -fmad=false), so
// the tensors are bit-identical to NumPy's.
#pragma once
#include "fot_device.cuh"

namespace fot {

// np.isclose(a, b) with the default rtol = 1e-5, atol = 1e-8, equal_nan = False
__device__ __forceinline__ bool np_isclose(double a, double b) {
  if (isfinite(a) && isfinite(b)) return fabs(a - b) <= 1e-8 + 1e-5 * fabs(b);
  return a == b;
}

// integrated_simulator.py:506-513: the current positions are prepended unless the prediction's first
// step already equals them for EVERY pedestrian (np.allclose).  Block-wide decision for one (query, sample).
__device__ __forceinline__ bool block_needs_prepend(const double* first_xy, int first_stride, const double* cur, int P) {
  __shared__ int s_differs;
  if (threadIdx.x == 0) s_differs = 0;
  __syncthreads();
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    const double fx = first_xy[(size_t)p * first_stride], fy = first_xy[(size_t)p * first_stride + 1];
    if (!(np_isclose(fx, cur[2 * p]) && np_isclose(fy, cur[2 * p + 1]))) s_differs = 1;
  }
  __syncthreads();
  const bool r = s_differs != 0;
  __syncthreads();
  return r;
}

// One block per query.  out[q][p][k][:]:  k = 0 the current position (when prepended), then
// current_pos + velocities * (time_target[i] + staleness).  When the prepend is skipped the tensor is one
// step shorter in the reference; the last step is then duplicated, which is what the sweep's time-index
// clamp (frenet_planner.py:1226-1227) makes of the shorter tensor.
__global__ void fot_cv_kernel(const double* __restrict__ p_curr, const double* __restrict__ p_prev,
                              const double* __restrict__ staleness, const double* __restrict__ time_target,
                              const double* __restrict__ cur_pos, double* __restrict__ out, int P, int n_steps,
                              int T_out, double sgan_dt, int obs_float32) {
  const int q = blockIdx.x;
  const double* pc = p_curr + (size_t)q * P * 2;
  const double* pp = p_prev ? p_prev + (size_t)q * P * 2 : nullptr;
  const double* cur = cur_pos ? cur_pos + (size_t)q * P * 2 : nullptr;
  double* o = out + (size_t)q * P * T_out * 2;
  const double stale = staleness ? staleness[q] : 0.0;
  const double t0 = time_target[0] + stale;
  extern __shared__ double s_first[];                   // [P][2] first predicted step
  // obs_float32: the simulator hands the predictor float32 observation tensors (observer.py:131-132), so the
  // positions are float32 values and the velocity is a float32 difference divided by float32(sgan_dt); the
  // extrapolation itself is float64 (NumPy promotes float32 * float64-scalar to float64).
  auto base = [&](int e) { return obs_float32 ? (double)(float)pc[e] : pc[e]; };
  auto vel = [&](int e) {
    if (!pp) return 0.0;
    if (obs_float32) return (double)(((float)pc[e] - (float)pp[e]) / (float)sgan_dt);
    return (pc[e] - pp[e]) / sgan_dt;                                 // :211
  };
  for (int e = threadIdx.x; e < 2 * P; e += blockDim.x) s_first[e] = base(e) + vel(e) * t0;
  __syncthreads();
  const bool prepend = cur && block_needs_prepend(s_first, 2, cur, P);
  const int shift = prepend ? 1 : 0;
  for (int idx = threadIdx.x; idx < P * T_out; idx += blockDim.x) {
    const int p = idx / T_out, k = idx - p * T_out;
    double x, y;
    if (k < shift) {
      x = cur[2 * p]; y = cur[2 * p + 1];
    } else {
      const int i = min(k - shift, n_steps - 1);
      const double t = time_target[i] + stale;                        // :225
      x = base(2 * p) + vel(2 * p) * t;                               // :226
      y = base(2 * p + 1) + vel(2 * p + 1) * t;
    }
    o[(size_t)idx * 2] = x;
    o[(size_t)idx * 2 + 1] = y;
  }
}

// np.interp(x, xp, fp) for one x (numpy/_core/src/multiarray/compiled_base.c arr_interp), xp increasing.
__device__ __forceinline__ double np_interp1(double x, const double* xp, const double* fp, int n) {
  if (x != x) return x;
  if (x > xp[n - 1]) return fp[n - 1];
  if (x < xp[0]) return fp[0];
  int lo = 0, hi = n - 1;                               // xp[lo] <= x, x <= xp[hi]; find j: xp[j] <= x < xp[j+1]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (x >= xp[mid]) lo = mid; else hi = mid;
  }
  int j = (x >= xp[n - 1]) ? n - 1 : lo;
  if (j == n - 1) return fp[j];
  if (xp[j] == x) return fp[j];
  const double slope = (fp[j + 1] - fp[j]) / (xp[j + 1] - xp[j]);
  double r = slope * (x - xp[j]) + fp[j];
  if (r != r) {
    r = slope * (x - xp[j + 1]) + fp[j + 1];
    if (r != r && fp[j] == fp[j + 1]) r = fp[j];
  }
  return r;
}

constexpr int kPredLenMax = 64;     // raw prediction steps (+ anchor) held per thread

// One block per (query, sample); one thread per (pedestrian, axis) coordinate series.
// pred [n_q][S][pred_len][P][2] (the predictor's own layout), anchor [n_q][P][2] or null;
// out [n_q][S][P][n_steps][2].
__global__ void fot_resample_kernel(const double* __restrict__ pred, const double* __restrict__ anchor,
                                    const double* __restrict__ staleness, const double* __restrict__ time_target,
                                    double* __restrict__ out, int S, int P, int pred_len, int n_steps, double sgan_dt) {
  const int q = blockIdx.x / S, sidx = blockIdx.x - q * S;
  const double* pr = pred + ((size_t)q * S + sidx) * pred_len * P * 2;
  const double* an = anchor ? anchor + (size_t)q * P * 2 : nullptr;
  double* o = out + ((size_t)q * S + sidx) * P * n_steps * 2;
  const double stale = staleness ? staleness[q] : 0.0;
  const int L = pred_len + (an ? 1 : 0);
  for (int e = threadIdx.x; e < 2 * P; e += blockDim.x) {
    const int p = e >> 1, ax = e & 1;
    double xs[kPredLenMax + 1], ys[kPredLenMax + 1];
    int n = 0;                                                         // source times relative to the current time (:271-275)
    if (an) { xs[0] = -stale; ys[0] = an[e]; n = 1; }
    for (int k = 1; k <= pred_len; ++k, ++n) {
      xs[n] = (double)k * sgan_dt - stale;
      ys[n] = pr[((size_t)(k - 1) * P + p) * 2 + ax];
    }
    bool all_first = true, all_zero = true;                            // :297 np.allclose(coords, coords[0]) / (coords, 0.0)
    for (int k = 0; k < L; ++k) {
      all_first &= np_isclose(ys[k], ys[0]);
      all_zero &= np_isclose(ys[k], 0.0);
    }
    const bool constant = all_first || all_zero;
    double v_tail = 0.0;
    if (!constant && L >= 2) {                                         // :305-311
      const int lookback = min(3, L);
      v_tail = (ys[L - 1] - ys[L - lookback]) / ((double)(lookback - 1) * sgan_dt);
      // Python's max(min(v_tail, 2.5), -2.5): a NaN passes through (fmin / fmax would drop it)
      v_tail = (2.5 < v_tail) ? 2.5 : v_tail;
      v_tail = (-2.5 > v_tail) ? -2.5 : v_tail;
    }
    double* row = o + (size_t)p * n_steps * 2 + ax;
    for (int i = 0; i < n_steps; ++i) {
      double v;
      const double t = time_target[i];
      if (constant) v = ys[L - 1];                                     // :298
      else if (L >= 2 && t > xs[L - 1]) v = ys[L - 1] + v_tail * (t - xs[L - 1]);   // :313-317
      else v = np_interp1(t, xs, ys, L);                               // :302
      row[(size_t)i * 2] = v;
    }
  }
}

// The t = 0 prepend (integrated_simulator.py:503-525).  in [n_q][S_in][P][T][2]; out [n_q][S_out][P][T+1][2]
// with S_out = 1 when `pick` selects one sample per query (the representative sample), else S_in.
// conditional != 0: the single-sample rule (:506-513, skip when the first step already equals the current
// positions for every pedestrian; the tensor is then one step shorter in the reference, here its last step
// is duplicated, which is what the sweep's time-index clamp makes of the shorter tensor);
// conditional == 0: the distribution rule (:517-525, always prepend).
__global__ void fot_prepend_kernel(const double* __restrict__ in, const int32_t* __restrict__ pick,
                                   const double* __restrict__ cur_pos, double* __restrict__ out, int S_in, int P, int T,
                                   int conditional) {
  const int S_out = pick ? 1 : S_in;
  const int q = blockIdx.x / S_out, so = blockIdx.x - q * S_out;
  const int si = pick ? pick[q] : so;
  const double* src = in + ((size_t)q * S_in + si) * P * T * 2;
  const double* cur = cur_pos + (size_t)q * P * 2;
  double* o = out + ((size_t)q * S_out + so) * P * (T + 1) * 2;
  const bool prepend = conditional ? block_needs_prepend(src, T * 2, cur, P) : true;
  for (int idx = threadIdx.x; idx < P * (T + 1); idx += blockDim.x) {
    const int p = idx / (T + 1), k = idx - p * (T + 1);
    double x, y;
    if (prepend) {
      if (k == 0) { x = cur[2 * p]; y = cur[2 * p + 1]; }
      else { x = src[((size_t)p * T + k - 1) * 2]; y = src[((size_t)p * T + k - 1) * 2 + 1]; }
    } else {
      const int kk = min(k, T - 1);
      x = src[((size_t)p * T + kk) * 2]; y = src[((size_t)p * T + kk) * 2 + 1];
    }
    o[(size_t)idx * 2] = x;
    o[(size_t)idx * 2 + 1] = y;
  }
}

// Closest-to-mean sample (trajectory_predictor.py:346-351): mean over the samples (sequential add over S,
// then / S, as np.mean reduces an outer axis), per-point 2-norm, np.sum over (pedestrians, steps) in NumPy's
// pairwise order, first arg-min.  fot_best_dist_kernel: one thread per (query, sample) distance;
// fot_best_pick_kernel: one thread per query picks the sample.
__global__ void fot_best_dist_kernel(const double* __restrict__ samples, double* __restrict__ dist, int n_q, int S, int PT) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_q * S) return;
  const int q = g / S, sidx = g - q * S;
  const double* base = samples + (size_t)q * S * PT * 2;
  const double* mine = base + (size_t)sidx * PT * 2;
  auto term = [&](int e) {
    double mx = base[(size_t)e * 2], my = base[(size_t)e * 2 + 1];
    for (int s2 = 1; s2 < S; ++s2) { mx += base[((size_t)s2 * PT + e) * 2]; my += base[((size_t)s2 * PT + e) * 2 + 1]; }
    mx = mx / (double)S; my = my / (double)S;
    const double dx = mine[(size_t)e * 2] - mx, dy = mine[(size_t)e * 2 + 1] - my;
    return sqrt(dx * dx + dy * dy);
  };
  dist[g] = np_pairwise_sum_flat(term, PT);
}
__global__ void fot_best_pick_kernel(const double* __restrict__ dist, int32_t* __restrict__ best_idx, int n_q, int S) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q < n_q) {
    int b = 0;                                          // np.argmin: first minimum, a NaN counts as the minimum
    for (int s2 = 1; s2 < S; ++s2) {
      const double cur_b = dist[(size_t)q * S + b], d = dist[(size_t)q * S + s2];
      if (cur_b != cur_b) break;
      if (d < cur_b || d != d) b = s2;
    }
    best_idx[q] = b;
  }
}

// ---- safety metrics (SURVEY.md section 8f, rank 2) -----------------------------------------------------
// compute_safety_metrics_static (src/core/data_structures.py:301-388): per query the minimum distance from
// any footprint circle centre to any pedestrian, the collision flag, the time to collision along the line
// of sight, the clearance and the clearance restricted to pedestrians ahead of the vehicle.  These are the
// inputs of the fail-safe state machine, needed once per query and step in batched roll-outs.
// One warp per query; out[q] = {min_distance, collision, ttc, clearance, clearance_ahead}.
// The reference's dot products are BLAS calls; the kernel writes out the order OpenBLAS's x86-64 kernels use
// (pinned on the host by tests/test_prediction_host_order.py):
//   [1,2] @ [2] and np.dot of two 2-vectors   fma(a1, b1, a0 * b0)
//   [k,2] @ [2], k >= 2                       fma(a0, b0, a1 * b1)
//   np.linalg.norm of a 2-vector              sqrt(fma(a1, a1, a0 * a0))
// np.linalg.norm(..., axis=2) over the distance matrix is an element-wise reduce: sqrt(a0 * a0 + a1 * a1).
struct CircleOffsets {
  double v[FOT_MAX_CIRCLES];          // EgoFootprint.offsets, passed by value (a kernel parameter, no device buffer)
};
// np.min: a NaN anywhere makes the minimum NaN (fmin would drop it)
__device__ __forceinline__ double nan_min(double a, double b) { return (a != a || a < b) ? a : b; }
__global__ void fot_safety_kernel(const double* __restrict__ ego, const double* __restrict__ ped_pos,
                                  const double* __restrict__ ped_vel, const int32_t* __restrict__ n_peds,
                                  double* __restrict__ out, int n_q, int P, double combined_radius,
                                  const CircleOffsets offsets, int n_circ) {
  const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (q >= n_q) return;
  const double* e = ego + 5 * (size_t)q;
  const double x = e[0], y = e[1], yaw = e[2], v = e[3];
  const double hx = cos(yaw), hy = sin(yaw);                                   // :371-372 / footprint.py:44
  const double evx = v * hx, evy = v * hy;                                     // :350-351
  const int np_ = min(max(n_peds ? n_peds[q] : P, 0), P);
  const double inf = INFINITY;
  double dmin = inf, ttc = inf, dmin_ahead = inf;
  for (int p = lane; p < np_; p += 32) {
    const double px = ped_pos[((size_t)q * P + p) * 2], py = ped_pos[((size_t)q * P + p) * 2 + 1];
    const double vx = ped_vel[((size_t)q * P + p) * 2], vy = ped_vel[((size_t)q * P + p) * 2 + 1];
    const double ax = px - x, ay = py - y;                                     // :373-374, one row or a [k,2] matrix
    const bool ahead = (np_ == 1 ? fma(ay, hy, ax * hx) : fma(ax, hx, ay * hy)) > 0.0;
    for (int c = 0; c < (n_circ > 0 ? n_circ : 1); ++c) {
      const double2 cc = n_circ > 0 ? footprint_centre(x, y, hx, hy, offsets.v[c]) : make_double2(x, y);   // footprint.py:45
      const double rx = px - cc.x, ry = py - cc.y;
      const double dist = sqrt(rx * rx + ry * ry);                             // :337-339
      dmin = nan_min(dmin, dist);
      if (ahead) dmin_ahead = nan_min(dmin_ahead, dist);
      const double rvx = vx - evx, rvy = vy - evy;
      const double along = -fma(ry, rvy, rx * rvx) / (sqrt(fma(ry, ry, rx * rx)) + 1e-8);   // :358
      if (along > 1e-5) {
        const double t = (dist - combined_radius) / along;                     // :360
        if (t >= 0.0) ttc = fmin(ttc, t);
      }
    }
  }
  for (int off = 16; off > 0; off >>= 1) {
    dmin = nan_min(dmin, __shfl_xor_sync(0xffffffffu, dmin, off));
    ttc = fmin(ttc, __shfl_xor_sync(0xffffffffu, ttc, off));                  // never NaN (t >= 0 above)
    dmin_ahead = nan_min(dmin_ahead, __shfl_xor_sync(0xffffffffu, dmin_ahead, off));
  }
  if (lane == 0) {
    double* o = out + 5 * (size_t)q;
    o[0] = dmin;                                                               // inf without pedestrians (:343)
    o[1] = dmin < combined_radius ? 1.0 : 0.0;                                 // :345
    o[2] = ttc;
    o[3] = dmin - combined_radius;                                             // :385
    o[4] = dmin_ahead == inf ? inf : dmin_ahead - combined_radius;             // :375-376
  }
}

}  // namespace fot
