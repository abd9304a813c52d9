// fot_assess_cand.cuh -- candidate assessment (fot_assess_candidates, sm_100a; DESIGN.md section 4j): every generated
// candidate of every query, regenerated on chip and assessed as fot_assess_trajectories assesses a series block, without
// a series ever reaching HBM.
//
//   fot_assess_cand_nan : one warp per 32 pedestrian trajectories of a query: the bit "a NaN at some step" of each
//                         (the NaN rule of fot_assess), once per launch, into the handle's scratch
//   fot_assess_cand     : (query, part) per CTA, one candidate per thread at a time, consecutive candidates on
//                         consecutive lanes (so the lanes of a warp mostly share the sample count and with it the
//                         obstacle time index: every obstacle load is warp-uniform).  A thread walks its candidate's
//                         samples in order, regenerates t, x, y and yaw with regenerate()'s device functions and tests
//                         the sample's circle centres against the field at once.  The query's obstacle block is staged
//                         in shared memory when it fits.  Per obstacle sample s the thread keeps a threshold mask in
//                         shared memory; a field with more than kCandPass samples is taken kCandPass samples per pass,
//                         the candidate regenerated in each pass, and the passes merged in the flat-index order.
#pragma once
#include "fot_assess.cuh"
#include "fot_weights.cuh"

namespace fot {

constexpr int kCandThreads = 128;
constexpr int kCandPass = 32;              // obstacle samples s per pass
constexpr size_t kCandStageMax = 48 * 1024;   // largest obstacle block staged in shared memory

struct AssessCand {
  Assess A;                  // m = cand_stride; series, len and n_t are not used
  int32_t* keep;             // [n_q][stride] kept samples, or null
  const unsigned* nan_bits;  // [n_q][nan_words]: bit sp set = pedestrian trajectory sp = s * P + p has a NaN step
  int32_t nan_words;
  int32_t sc;                // obstacle samples per pass: min(S, kCandPass), 0 without dynamic obstacles
  int32_t cpq;               // CTAs per query
};

// Dynamic shared memory of fot_assess_cand: the time table, the staged obstacle block, per thread sc hit masks and the
// first hit sample and hit count per threshold pair.
__host__ __device__ constexpr size_t assess_cand_smem(int NT, int n_r, int sc, size_t stage_bytes) {
  return (size_t)kTT * NT * sizeof(double) + stage_bytes + (size_t)kCandThreads * (sc + 2 * n_r) * sizeof(unsigned);
}

__global__ void __launch_bounds__(256)
fot_assess_cand_nan(const double2* __restrict__ dyn, long long SP, int T, long long n_words_total, int words,
                    unsigned* __restrict__ bits) {
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n_words_total) return;
  const long long q = w / words, k = w - q * words;
  const double2* dq = dyn + (size_t)q * SP * T;
  unsigned word = 0;
  for (int j = 0; j < 32; ++j) {
    const long long sp = k * 32 + j;
    if (sp >= SP) break;
    bool bad = false;
    for (int e = lane; e < T; e += 32) bad |= nan_step(dq[sp * T + e]);
    if (__any_sync(0xffffffffu, bad)) word |= 1u << j;
  }
  if (lane == 0) bits[w] = word;
}

// B: the queries (frenet, v_grid, n_v, routes) and the field (dyn_raw null: no dynamic obstacles; static_raw null: no
// static points).  kStage: the query's [S][P][T_obs] block is copied to shared memory first.
template <bool kStage>
__global__ void __launch_bounds__(kCandThreads)
fot_assess_cand(const Plan P, const Batch B, const AssessCand C) {
  extern __shared__ __align__(16) unsigned char cand_sm[];
  const Assess& A = C.A;
  const int bd = blockDim.x, tid = threadIdx.x;
  const int q = blockIdx.x / C.cpq, part = blockIdx.x - q * C.cpq;
  const int n_r = A.n_r, NT = P.n_t_max, sc = C.sc;
  const int nc = P.cfg.n_circles > 0 ? P.cfg.n_circles : 1;
  const int S = B.dyn_raw ? B.S : 0, Pn = B.P, T = B.T_obs, M = B.static_raw ? B.n_static : 0;
  const long long SP = (long long)S * Pn;
  double* tt = reinterpret_cast<double*>(cand_sm);                                  // [NT][kTT]
  double2* sdyn = reinterpret_cast<double2*>(tt + (size_t)kTT * NT);                 // [S*P][T] (kStage)
  unsigned* msk = reinterpret_cast<unsigned*>(sdyn + (kStage ? SP * T : 0));        // [sc][bd] thresholds hit in sample s
  int* first = reinterpret_cast<int*>(msk + (size_t)sc * bd);                       // [n_r][bd] first sample with a hit
  int* cnt = first + (size_t)n_r * bd;                                               // [n_r][bd] obstacle samples hit
  __shared__ double s_r2d[FOT_MAX_RADII], s_r2s[FOT_MAX_RADII];

  const size_t o0 = (size_t)q * A.m;
  Plan V;                                                // the query's route; a bad id: every column blank
  const bool routed = route_plan(P, B.rt, q, V);
  int grid_total = 0;
  const int n_cand = routed ? weighted_candidates(P, B, q, &grid_total) : 0;
  for (int i = n_cand + part * bd + tid; i < A.m; i += C.cpq * bd) {               // columns past the candidates
    assess_blank(A, o0 + i);
    if (C.keep) C.keep[o0 + i] = 0;
  }
  if (n_cand == 0) return;                               // uniform over the block

  if (tid < n_r) { s_r2d[tid] = A.r2[2 * tid]; s_r2s[tid] = A.r2[2 * tid + 1]; }
  for (int n = tid; n < NT; n += bd) tt_fill(tt, n, P.cfg.dt);
  const double2* dynq = S > 0 ? reinterpret_cast<const double2*>(B.dyn_raw) + (size_t)q * SP * T : nullptr;
  if (kStage)
    for (long long e = tid; e < SP * T; e += bd) sdyn[e] = dynq[e];
  __syncthreads();
  double r2d_max = -INFINITY, r2s_max = -INFINITY;      // one comparison per distance in the common case
  for (int r = 0; r < n_r; ++r) { r2d_max = fmax(r2d_max, s_r2d[r]); r2s_max = fmax(r2s_max, s_r2s[r]); }
  const double* statq = M > 0 ? B.static_raw + (B.static_per_query ? (size_t)q * M * 2 : 0) : nullptr;
  const unsigned* nanq = S > 0 ? C.nan_bits + (size_t)q * C.nan_words : nullptr;
  const double* fs = B.frenet + 6 * (size_t)q;
  const int n_v = B.n_v[q], n_d = P.cfg.n_d;
  const int n_pass = S > 0 ? (S + sc - 1) / sc : 1;

  for (int i = part * bd + tid; i < n_cand; i += C.cpq * bd) {
    // ---- candidate i, decoded and solved as regenerate() does
    Lon lon;
    Lat lat;
    int N;
    if (i < grid_total) {
      const int id = i % n_d, kv = (i / n_d) % n_v, jT = i / (n_d * n_v);
      N = V.n_steps[jT] + 1;
      lon = lon_solve(fs, B.v_grid[(size_t)q * B.n_v_max + kv], V.T[jT], V.inv4 + 4 * jT, n_v == 1, N - 1);
      lat = lat_solve(fs, V.d_grid[id], V.T[jT], V.inv5 + 9 * jT, n_d == 1, N - 1);
    } else {
      const int bi = i - grid_total;
      N = V.cfg.n_total;
      lon = lon_solve(fs, 0.0, V.Tb[bi], V.inv4b + 4 * bi, true, V.n_steps_b[bi]);
      lat = lat_solve(fs, fs[3], V.Tb[bi], V.inv5b + 9 * bi, true, V.n_steps_b[bi]);
    }
    for (int r = 0; r < n_r; ++r) { first[r * bd + tid] = INT_MAX; cnt[r * bd + tid] = 0; }
    int fn = N;                                          // first sample with a NaN x (N: none)
    bool singular = false;                               // fp.py:826-833: some sample with a finite q <= 0.05
    double dmin = INFINITY, smin = INFINITY;
    long long dat = LLONG_MAX, sat = LLONG_MAX;
    unsigned shit = 0;
    for (int pass = 0; pass < n_pass; ++pass) {
      const int s0 = pass * sc, ns = S > 0 ? min(sc, S - s0) : 0;
      for (int j = 0; j < ns; ++j) msk[j * bd + tid] = 0;
      double pm = INFINITY;                              // this pass's dynamic minimum (visited in flat-index order)
      long long pat = LLONG_MAX;
      unsigned seen = 0;
      const int lim = pass == 0 ? N : fn;                // pass 0 looks at every sample for the singularity guard
      for (int n = 0; n < lim; ++n) {
        const double s = lon_p0(lon, tt, n), sd = lon_p1(lon, tt, n), sdd = lon_p2(lon, tt, n);
        const double d = lat_p0(lat, tt, n), dd = lat_p1(lat, tt, n), ddd = lat_p2(lat, tt, n);
        const RefPt rp = spline_ref(V, s);
        if (pass == 0) {
          const double qq = 1.0 - rp.rk * d;            // fp.py:826
          singular |= (qq <= 0.05) & (fabs(qq) < INFINITY);
        }
        if (n >= fn) continue;
        double sn, cs;
        sincos(rp.rth, &sn, &cs);
        const CartPt cp = to_cartesian(rp.rx, rp.ry, cs, sn, rp.rth, rp.rk, rp.rdk, sd, sdd, d, dd, ddd);
        if (cp.x != cp.x) { fn = n; continue; }
        // ---- sample n: its circle centres against the field, in the flat-index order of fot_assess
        const int kt = S > 0 ? obstacle_step(tt[kTT * n], P.cfg.dt, T) : 0;
        double hx = 0.0, hy = 0.0;
        if (P.cfg.n_circles > 0) {
          const double yaw = wrap_angle(cp.ang);
          hx = cos(yaw); hy = sin(yaw);
        }
        unsigned hn = 0;
        for (int c = 0; c < nc; ++c) {
          const double2 p = P.cfg.n_circles == 0 ? make_double2(cp.x, cp.y)
                                                 : footprint_centre(cp.x, cp.y, hx, hy, P.cfg.circle_offsets[c]);
          const long long f = (long long)n * nc + c;
          if (pass == 0) {
            for (int k = 0; k < M; ++k) {
              const double dx = p.x - statq[2 * k], dy = p.y - statq[2 * k + 1];
              const double d2 = dx * dx + dy * dy;
              if (d2 < smin || (d2 == smin && sat == LLONG_MAX)) { smin = d2; sat = f * M + k; }
              if (d2 <= r2s_max) { const unsigned h = radii_hit(s_r2s, n_r, d2); shit |= h; hn |= h; }
            }
          }
          for (int j = 0; j < ns; ++j) {
            const long long b0 = (long long)(s0 + j) * Pn;
            unsigned m = 0;
            for (int pp = 0; pp < Pn; ++pp) {
              const long long sp = b0 + pp;
              if ((__ldg(nanq + (sp >> 5)) >> (sp & 31)) & 1u) continue;     // the NaN rule (fp.py:1211-1222)
              const double2 o = kStage ? sdyn[sp * T + kt] : __ldg(dynq + sp * T + kt);
              const double dx = p.x - o.x, dy = p.y - o.y;
              const double d2 = dx * dx + dy * dy;
              if (d2 < pm || (d2 == pm && pat == LLONG_MAX)) { pm = d2; pat = f * SP + sp; }
              if (d2 <= r2d_max) m |= radii_hit(s_r2d, n_r, d2);
            }
            if (m) { msk[j * bd + tid] |= m; hn |= m; }
          }
        }
        for (unsigned nb = hn & ~seen; nb; nb &= nb - 1) {
          const int r = __ffs(nb) - 1;
          first[r * bd + tid] = min(first[r * bd + tid], n);
        }
        seen |= hn;
      }
      if (singular || fn < 2) break;                     // kept length 0 (fp.py:866): a blank entry
      argmin_merge(dmin, dat, pm, pat);
      for (int j = 0; j < ns; ++j) {
        const unsigned mk = msk[j * bd + tid];
        for (int r = 0; r < n_r; ++r) cnt[r * bd + tid] += (mk >> r) & 1u;
      }
    }

    // ---- the outputs of column i
    const size_t o = o0 + i;
    const int keep = (singular || fn < 2) ? 0 : fn;
    if (C.keep) C.keep[o] = keep;
    if (keep == 0) { assess_blank(A, o); continue; }
    A.dyn_min[o] = dat == LLONG_MAX ? INFINITY : sqrt(dmin);
    if (dat == LLONG_MAX) {
      for (int k = 0; k < 4; ++k) A.dyn_at[4 * o + k] = -1;
    } else {
      const long long per_n = (long long)nc * SP, rem = dat % per_n, sp = rem % SP;
      A.dyn_at[4 * o] = (int)(dat / per_n); A.dyn_at[4 * o + 1] = (int)(rem / SP);
      A.dyn_at[4 * o + 2] = (int)(sp / Pn); A.dyn_at[4 * o + 3] = (int)(sp % Pn);
    }
    A.static_min[o] = sat == LLONG_MAX ? INFINITY : sqrt(smin);
    if (sat == LLONG_MAX) {
      for (int k = 0; k < 3; ++k) A.static_at[3 * o + k] = -1;
    } else {
      const long long per_n = (long long)nc * M, rem = sat % per_n;
      A.static_at[3 * o] = (int)(sat / per_n); A.static_at[3 * o + 1] = (int)(rem / M); A.static_at[3 * o + 2] = (int)(rem % M);
    }
    for (int r = 0; r < n_r; ++r) {
      const int fh = first[r * bd + tid];
      A.dyn_hits[o * n_r + r] = cnt[r * bd + tid];
      A.first_hit[o * n_r + r] = fh == INT_MAX ? -1 : fh;
      A.static_hit[o * n_r + r] = (int)((shit >> r) & 1u);
    }
  }
}

}  // namespace fot
