// fot_rank.cuh -- ranked alternatives: the k best feasible candidates of every query (fot_rank_candidates, sm_100a).
//
//   fot_rank        : one block per query.  From the per-candidate table a sweep launch wrote (cand_cat / cand_cost),
//                     the k smallest (cost, index) pairs among the candidates the winner selection could pick:
//                     category FOT_CAT_OK and cost < +inf (a NaN or infinite cost never wins, fp.py:1254-1257).
//   fot_rank_series : one block per (query, rank) that holds a candidate: its 15 series and kept length, regenerated
//                     by the same device function as fot_winner's.
#pragma once
#include "fot_kernels.cuh"

namespace fot {

constexpr int kRankThreads = 256;

struct Ranked {
  int32_t k;
  int32_t* idx; double* cost; int32_t* len; double* series;
};

// k rounds of a block-wide arg-min over the entries strictly after the previous round's winner in (cost, index)
// order -- the comparator of argmin_merge, so rank 0 is the winner of the same launch.  Every round is an exact
// minimum, whatever the thread count; the row (1261 candidates, 11 KB, in config 4) stays in L1 between rounds.
__global__ void __launch_bounds__(kRankThreads)
fot_rank(const uint8_t* __restrict__ cand_cat, const double* __restrict__ cand_cost, int stride, const Ranked R) {
  __shared__ double s_cost[kRankThreads / 32];
  __shared__ int s_idx[kRankThreads / 32];
  const int q = blockIdx.x, tid = threadIdx.x;
  const uint8_t* cat = cand_cat + (size_t)q * stride;
  const double* cost = cand_cost + (size_t)q * stride;
  double pc = -INFINITY;
  int pi = -1;
  int r = 0;
  for (; r < R.k; ++r) {
    double c = INFINITY;
    int i = 0x7fffffff;
    for (int j = tid; j < stride; j += kRankThreads) {
      if (cat[j] != FOT_CAT_OK) continue;
      const double v = cost[j];
      if (v < INFINITY && (v > pc || (v == pc && j > pi))) argmin_merge(c, i, v, j);
    }
    for (int off = 16; off > 0; off >>= 1) {
      const double oc = __shfl_down_sync(0xffffffffu, c, off);
      const int oi = __shfl_down_sync(0xffffffffu, i, off);
      argmin_merge(c, i, oc, oi);
    }
    if ((tid & 31) == 0) { s_cost[tid >> 5] = c; s_idx[tid >> 5] = i; }
    __syncthreads();
    c = s_cost[0]; i = s_idx[0];
    for (int w = 1; w < kRankThreads / 32; ++w) argmin_merge(c, i, s_cost[w], s_idx[w]);
    __syncthreads();                                   // the next round overwrites s_cost / s_idx
    if (i == 0x7fffffff) break;                        // no further feasible candidate (uniform over the block)
    if (tid == 0) { R.idx[(size_t)q * R.k + r] = i; R.cost[(size_t)q * R.k + r] = c; }
    pc = c; pi = i;
  }
  for (int p = r + tid; p < R.k; p += kRankThreads) {
    R.idx[(size_t)q * R.k + p] = -1;
    R.cost[(size_t)q * R.k + p] = INFINITY;
    if (R.len) R.len[(size_t)q * R.k + p] = 0;
  }
}

// Behind fot_rank in stream order.  R.len is not null here; R.series may be (lengths only).
__global__ void __launch_bounds__(128)
fot_rank_series(const Plan P, const Batch B, const Ranked R) {
  extern __shared__ double sm[];
  double* tt = sm;   // [NT][kTT]
  __shared__ int s_first_nan;
  const int NT = P.n_t_max;
  const size_t slot = blockIdx.x;                      // q * k + rank
  const int i = R.idx[slot];
  if (i < 0) return;
  const int q = (int)(slot / R.k);
  Plan V;                                              // the query's route (a bad id never ranks a candidate)
  if (!route_plan(P, B.rt, q, V)) return;
  if (threadIdx.x == 0) s_first_nan = 0x7fffffff;
  for (int n = threadIdx.x; n < NT; n += blockDim.x) tt_fill(tt, n, P.cfg.dt);
  __syncthreads();
  const int len = R.series ? regenerate<true>(V, B, q, i, tt, R.series + slot * FOT_N_SERIES * NT, nullptr, &s_first_nan)
                           : regenerate<false>(V, B, q, i, tt, nullptr, nullptr, &s_first_nan);
  if (threadIdx.x == 0) R.len[slot] = len;
}

}  // namespace fot
