// fot_assess.cuh -- trajectory assessment (fot_assess_trajectories, sm_100a; DESIGN.md section 4i): for m given
// trajectories per query, the closest approach to an obstacle field and the collision counts under n_r radii, in the
// reference's collision geometry (fp.py:1126-1233).  Reads only the series rows t, x, y and yaw.
//
// One block per query.  The block takes the query's trajectories in chunks of at most blockDim samples (whole
// trajectories: blockDim >= the row length), one sample per thread, and stages the chunk's circle centres in shared
// memory.  It then streams the obstacle tensor once per chunk -- once per query whenever the chunk holds every
// trajectory, as it does for winners and ranked alternatives -- 32 pedestrian trajectories at a time: the block first
// reads the 32 trajectories in full (consecutive threads take consecutive time steps, one contiguous stretch of
// memory) to find those with a NaN anywhere, then every thread tests its own sample against the others' positions at
// its time index, loads that coalesce across the lanes' consecutive samples and hit L1.
#pragma once
#include "fot_kernels.cuh"

namespace fot {

constexpr int kAssessMaxThreads = 512;     // >= FOT_MAX_ASSESS_NT: a trajectory never straddles two chunks
static_assert(FOT_MAX_ASSESS_NT <= kAssessMaxThreads, "a chunk must hold the longest trajectory");
constexpr int kSeriesT = 0, kSeriesX = 9, kSeriesY = 10, kSeriesYaw = 11;   // rows of the series block (SERIES order)

struct Assess {
  int32_t m, n_t, n_r;
  const double* series; const int32_t* len; const double* r2;
  double* dyn_min; int32_t* dyn_at; double* static_min; int32_t* static_at;
  int32_t* dyn_hits; int32_t* first_hit; int32_t* static_hit;
};

// Bytes of dynamic shared memory per thread: the sample's n_circ centres and its five partial results.
__host__ __device__ constexpr size_t assess_smem_per_thread(int n_circ) {
  return (size_t)n_circ * sizeof(double2) + 2 * sizeof(double) + 2 * sizeof(long long) + 2 * sizeof(unsigned);
}

// Obstacle time index of a sample at time t: clip(rint(t / dt), 0, T_obs - 1) (fp.py:1226-1227).  A NaN or infinite
// t gives 0, as NumPy's cast of it to an integer (the smallest int64) clipped does.
__device__ __forceinline__ int obstacle_step(double t, double dt, int T_obs) {
  const double k = rint(t / dt);
  if (!(k >= 0.0) || k == INFINITY) return 0;
  return k >= (double)(T_obs - 1) ? T_obs - 1 : (int)k;
}

// The thresholds r2[0 .. n_r) that a squared distance is within, as a bit mask (a NaN d2 is within none).
__device__ __forceinline__ unsigned radii_hit(const double* r2, int n_r, double d2) {
  unsigned m = 0;
  for (int r = 0; r < n_r; ++r)
    if (d2 <= r2[r]) m |= 1u << r;
  return m;
}

__device__ __forceinline__ void assess_blank(const Assess& A, size_t o) {
  A.dyn_min[o] = INFINITY; A.static_min[o] = INFINITY;
  for (int k = 0; k < 4; ++k) A.dyn_at[4 * o + k] = -1;
  for (int k = 0; k < 3; ++k) A.static_at[3 * o + k] = -1;
  for (int r = 0; r < A.n_r; ++r) {
    A.dyn_hits[o * A.n_r + r] = 0; A.first_hit[o * A.n_r + r] = -1; A.static_hit[o * A.n_r + r] = 0;
  }
}

// B: the obstacle field (dyn_raw null: no dynamic obstacles; static_raw null: no static points).
__global__ void __launch_bounds__(kAssessMaxThreads)
fot_assess(const Plan P, const Batch B, const Assess A) {
  extern __shared__ __align__(16) unsigned char assess_sm[];
  double* sm = reinterpret_cast<double*>(assess_sm);
  const int bd = blockDim.x, tid = threadIdx.x, q = blockIdx.x;
  const int nc = P.cfg.n_circles > 0 ? P.cfg.n_circles : 1;
  double2* cen = reinterpret_cast<double2*>(sm);                  // [nc][bd] circle centres of the chunk's samples
  double* sl_dmin = sm + 2 * (size_t)nc * bd;                     // [bd] per sample: closest dynamic d2,
  double* sl_smin = sl_dmin + bd;                                 //      closest static d2,
  long long* sl_dat = reinterpret_cast<long long*>(sl_smin + bd); //      their flat indices,
  long long* sl_sat = sl_dat + bd;
  unsigned* sl_hit = reinterpret_cast<unsigned*>(sl_sat + bd);    //      thresholds hit by any obstacle,
  unsigned* sl_shit = sl_hit + bd;                                //      thresholds hit by a static point
  __shared__ double s_r2d[FOT_MAX_RADII], s_r2s[FOT_MAX_RADII];
  __shared__ int s_j[kAssessMaxThreads], s_off[kAssessMaxThreads + 1];
  __shared__ unsigned s_smask[kAssessMaxThreads];                 // per chunk trajectory: thresholds hit in sample s
  __shared__ unsigned s_nan[2];                                   // NaN trajectories of a group of 32 (double-buffered)
  __shared__ int s_nj, s_next;

  const int n_r = A.n_r;
  if (tid < n_r) { s_r2d[tid] = A.r2[2 * tid]; s_r2s[tid] = A.r2[2 * tid + 1]; }
  for (int i = tid; i < bd; i += bd) s_smask[i] = 0;
  __syncthreads();
  double r2d_max = -INFINITY, r2s_max = -INFINITY;               // one comparison per distance in the common case
  for (int r = 0; r < n_r; ++r) { r2d_max = fmax(r2d_max, s_r2d[r]); r2s_max = fmax(r2s_max, s_r2s[r]); }

  const int S = B.dyn_raw ? B.S : 0, Pn = B.P, T = B.T_obs, M = B.static_raw ? B.n_static : 0;
  const long long SP = (long long)S * Pn;
  const double2* dynq = S > 0 ? reinterpret_cast<const double2*>(B.dyn_raw) + (size_t)q * SP * T : nullptr;
  const double* statq = M > 0 ? B.static_raw + (B.static_per_query ? (size_t)q * M * 2 : 0) : nullptr;
  const size_t qm = (size_t)q * A.m;
  const size_t NT = (size_t)A.n_t;

  for (int j0 = 0;;) {
    // ---- the next chunk: whole trajectories, at most bd samples; empty slots get blank outputs here
    if (tid == 0) {
      int n = 0, cnt = 0, j = j0;
      for (; j < A.m; ++j) {
        const int L = min(max(A.len[qm + j], 0), A.n_t);
        if (L == 0) { assess_blank(A, qm + j); continue; }
        if (n + L > bd) break;
        s_j[cnt] = j; s_off[cnt] = n; n += L; ++cnt;
      }
      s_off[cnt] = n; s_nj = cnt; s_next = j;
      s_nan[0] = s_nan[1] = 0;
    }
    __syncthreads();
    const int nj = s_nj, n_items = s_off[nj], next = s_next;
    if (nj == 0) break;

    // ---- this thread's sample (jl, n) and its circle centres
    const bool act = tid < n_items;
    int jl = 0, n = 0, kt = 0;
    if (act) {
      int lo = 0, hi = nj - 1;
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (s_off[mid] <= tid) lo = mid; else hi = mid - 1;
      }
      jl = lo; n = tid - s_off[jl];
      const double* row = A.series + (qm + s_j[jl]) * FOT_N_SERIES * NT + n;
      const double x = row[kSeriesX * NT], y = row[kSeriesY * NT];
      if (S > 0) kt = obstacle_step(row[kSeriesT * NT], P.cfg.dt, T);
      if (P.cfg.n_circles == 0) {
        cen[tid] = make_double2(x, y);
      } else {
        const double yaw = row[kSeriesYaw * NT];
        const double hx = cos(yaw), hy = sin(yaw);
        for (int c = 0; c < nc; ++c) cen[(size_t)c * bd + tid] = footprint_centre(x, y, hx, hy, P.cfg.circle_offsets[c]);
      }
    }
    const long long flat_n = (long long)n * nc;                  // (n, c) prefix of the flat indices

    // ---- static points: flat index over [len, n_circ, M]
    double smin = INFINITY, dmin = INFINITY;
    long long sat = LLONG_MAX, dat = LLONG_MAX;
    unsigned shit = 0, hit = 0;
    if (act && statq) {
      for (int k = 0; k < M; ++k) {
        const double ox = statq[2 * k], oy = statq[2 * k + 1];
        for (int c = 0; c < nc; ++c) {
          const double2 p = cen[(size_t)c * bd + tid];
          const double dx = p.x - ox, dy = p.y - oy;
          const double d2 = dx * dx + dy * dy;
          argmin_merge(smin, sat, d2, (flat_n + c) * M + k);
          if (d2 <= r2s_max) shit |= radii_hit(s_r2s, n_r, d2);
        }
      }
    }

    // ---- dynamic obstacles: flat index over [len, n_circ, S, P]; per sample s, which thresholds some entry hits
    int cnt[FOT_MAX_RADII];
#pragma unroll
    for (int r = 0; r < FOT_MAX_RADII; ++r) cnt[r] = 0;
    int it = 0;
    for (int s = 0; s < S; ++s) {
      unsigned smask = 0;
      for (int p0 = 0; p0 < Pn; p0 += 32, ++it) {
        const int np_ = min(32, Pn - p0);
        const double2* grp = dynq + ((size_t)s * Pn + p0) * T;    // 32 trajectories, contiguous
        unsigned* nanw = &s_nan[it & 1];
        for (long long e = tid; e < (long long)np_ * T; e += bd)
          if (nan_step(grp[e])) atomicOr(nanw, 1u << (int)(e / T));
        __syncthreads();
        const unsigned bad = *nanw;
        if (tid == 0) s_nan[(it & 1) ^ 1] = 0;                    // the next group's word; last read a group ago
        if (act) {
          for (int pp = 0; pp < np_; ++pp) {
            if ((bad >> pp) & 1u) continue;                       // a NaN anywhere: the trajectory is ignored (fp.py:1211-1222)
            const double2 o = grp[(size_t)pp * T + kt];
            const long long f = (long long)s * Pn + p0 + pp;
            for (int c = 0; c < nc; ++c) {
              const double2 p = cen[(size_t)c * bd + tid];
              const double dx = p.x - o.x, dy = p.y - o.y;
              const double d2 = dx * dx + dy * dy;
              argmin_merge(dmin, dat, d2, (flat_n + c) * SP + f);
              if (d2 <= r2d_max) smask |= radii_hit(s_r2d, n_r, d2);
            }
          }
        }
        __syncthreads();
      }
      if (smask) { atomicOr(&s_smask[jl], smask); hit |= smask; }
      __syncthreads();
      if (tid < nj) {
        const unsigned mk = s_smask[tid];
        s_smask[tid] = 0;
#pragma unroll
        for (int r = 0; r < FOT_MAX_RADII; ++r) cnt[r] += (mk >> r) & 1u;
      }
      __syncthreads();
    }

    // ---- per trajectory: merge its samples in sample order (thread jl owns trajectory jl of the chunk)
    if (act) {
      sl_dmin[tid] = dmin; sl_dat[tid] = dat; sl_smin[tid] = smin; sl_sat[tid] = sat;
      sl_hit[tid] = hit | shit; sl_shit[tid] = shit;
    }
    __syncthreads();
    if (tid < nj) {
      const size_t o = qm + s_j[tid];
      const int a = s_off[tid], b = s_off[tid + 1];
      double dm = INFINITY, sm2 = INFINITY;
      long long di = LLONG_MAX, si = LLONG_MAX;
      unsigned sh = 0;
      for (int i = a; i < b; ++i) {
        argmin_merge(dm, di, sl_dmin[i], sl_dat[i]);
        argmin_merge(sm2, si, sl_smin[i], sl_sat[i]);
        sh |= sl_shit[i];
      }
      A.dyn_min[o] = di == LLONG_MAX ? INFINITY : sqrt(dm);
      if (di == LLONG_MAX) {
        for (int k = 0; k < 4; ++k) A.dyn_at[4 * o + k] = -1;
      } else {
        const long long per_n = (long long)nc * SP, rem = di % per_n, sp = rem % SP;
        A.dyn_at[4 * o] = (int)(di / per_n); A.dyn_at[4 * o + 1] = (int)(rem / SP);
        A.dyn_at[4 * o + 2] = (int)(sp / Pn); A.dyn_at[4 * o + 3] = (int)(sp % Pn);
      }
      A.static_min[o] = si == LLONG_MAX ? INFINITY : sqrt(sm2);
      if (si == LLONG_MAX) {
        for (int k = 0; k < 3; ++k) A.static_at[3 * o + k] = -1;
      } else {
        const long long per_n = (long long)nc * M, rem = si % per_n;
        A.static_at[3 * o] = (int)(si / per_n); A.static_at[3 * o + 1] = (int)(rem / M); A.static_at[3 * o + 2] = (int)(rem % M);
      }
#pragma unroll
      for (int r = 0; r < FOT_MAX_RADII; ++r) {
        if (r >= n_r) continue;                                   // (not break: cnt[] stays in registers)
        int first = -1;
        for (int i = a; i < b; ++i)
          if ((sl_hit[i] >> r) & 1u) { first = i - a; break; }
        A.dyn_hits[o * n_r + r] = cnt[r];
        A.first_hit[o * n_r + r] = first;
        A.static_hit[o * n_r + r] = (int)((sh >> r) & 1u);
      }
    }
    __syncthreads();                                              // s_j / s_off / slots are the next chunk's
    if (next >= A.m) break;
    j0 = next;
  }
}

}  // namespace fot
