// fot_kernels.cuh -- the launch-level kernels around the sweep (sm_100a, fp64).  The sweep kernels themselves are in
// fot_sweep_items.cuh and fot_sweep_pairs.cuh, their shared per-candidate arithmetic in fot_sweep_math.cuh.
//
//   fot_init_kernel : per launch, zero the histogram and mark every per-candidate category unwritten
//   fot_prepass : per launch, the cost tables (jerk sums, terminal offsets) and the predicted trajectories' boxes
//   fot_winner : per query, reduce the sweep's per-CTA partials and regenerate the 15 sequences of the
//        winning candidate only, in the reference's arithmetic order.
#pragma once
#include "fot_device.cuh"

namespace fot {

// flag bits of the priority chain fp.py:964-991
enum : unsigned { F_SPEED = 1u, F_ACCEL = 2u, F_CURV = 4u, F_LAT = 8u, F_ROAD = 16u };

// Per-launch initialisation (kept off the copy engines, which cudaMemsetAsync may use and which are
// busy with the next chunk's upload in the pipelined host path).
__global__ void fot_init_kernel(int32_t* stats, int n_stats, uint8_t* cand_cat, size_t n_cat) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = i; j < (size_t)n_stats; j += stride) stats[j] = 0;
  for (size_t j = i; j < n_cat; j += stride) cand_cat[j] = FOT_CAT_DROP + 1;
}

// ---- TMA / mbarrier helpers (cp.async.bulk global -> shared, completion on an mbarrier) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// Cost pieces that depend on one polynomial profile only (fp.py:703-734): the jerk sums  sum_n s'''(t_n)^2,
// sum_n d'''(t_n)^2  in NumPy's pairwise-summation order (so that costs are bit-identical to the
// reference) and the terminal lateral offset d(t_end).  One thread per profile; per query the table holds
//   [n_T][n_v_max] Js | [n_T][n_d] Jp | [n_T][n_d] d_end | [n_B] Js brake | [n_B] Jp brake | [n_B] d_end brake.
__device__ __forceinline__ void cost_prepass_body(const Plan& P, const Batch& B, double* __restrict__ tab, unsigned block) {
  const int n_d = P.cfg.n_d, n_T = P.cfg.n_T, n_B = P.cfg.n_B;
  const int nTv = n_T * B.n_v_max, nTd = n_T * n_d;
  const int n_prof = nTv + nTd + 2 * n_B;                // profiles with a sum
  const int stride = nTv + 2 * nTd + 3 * n_B;
  const long long g = (long long)block * blockDim.x + threadIdx.x;    // one thread per profile
  if (g >= (long long)B.n_q * n_prof) return;
  const int q = (int)(g / n_prof), pr = (int)(g - (long long)q * n_prof);
  const double* fs = B.frenet + 6 * (size_t)q;
  const double dt = P.cfg.dt;
  double* out = tab + (size_t)q * stride;
  const int n_v = B.n_v[q];
  if (pr < nTv || (pr >= nTv + nTd && pr < nTv + nTd + n_B)) {             // longitudinal
    Lon L;
    int N, slot;
    if (pr < nTv) {
      const int jT = pr / B.n_v_max, kv = pr - jT * B.n_v_max;
      if (kv >= n_v) return;
      N = P.n_steps[jT] + 1;
      L = lon_solve(fs, B.v_grid[(size_t)q * B.n_v_max + kv], P.T[jT], P.inv4 + 4 * jT, n_v == 1, N - 1);
      slot = pr;
    } else {
      const int b = pr - nTv - nTd;
      N = P.cfg.n_total;
      L = lon_solve(fs, 0.0, P.Tb[b], P.inv4b + 4 * b, true, P.n_steps_b[b]);
      slot = nTv + 2 * nTd + b;
    }
    const double a3 = L.a3, a4 = L.a4;
    const int hold = L.hold;
    auto jerk2 = [=](int k) {                            // fp.py:647, :722
      const double j = k > hold ? 0.0 : 6.0 * a3 + 24.0 * a4 * ((double)k * dt);
      return j * j;
    };
    out[slot] = np_pairwise_sum_flat(jerk2, N);
  } else {                                               // lateral
    Lat L;
    int N, slot_j, slot_d;
    if (pr < nTv + nTd) {
      const int li = pr - nTv, jT = li / n_d, id = li - jT * n_d;
      N = P.n_steps[jT] + 1;
      L = lat_solve(fs, P.d_grid[id], P.T[jT], P.inv5 + 9 * jT, n_d == 1, N - 1);
      slot_j = nTv + li; slot_d = nTv + nTd + li;
    } else {
      const int b = pr - nTv - nTd - n_B;
      N = P.cfg.n_total;
      L = lat_solve(fs, fs[3], P.Tb[b], P.inv5b + 9 * b, true, P.n_steps_b[b]);
      slot_j = nTv + 2 * nTd + n_B + b; slot_d = nTv + 2 * nTd + 2 * n_B + b;
    }
    const double a3 = L.a3, a4 = L.a4, a5 = L.a5;
    const int hold = L.hold;
    auto jerk2 = [=](int k) {                            // fp.py:691, :718
      const double t = (double)k * dt;
      const double j = k > hold ? 0.0 : 6.0 * a3 + 24.0 * a4 * t + 60.0 * a5 * (t * t);
      return j * j;
    };
    out[slot_j] = np_pairwise_sum_flat(jerk2, N);
    const TPow te = tpow(min(N - 1, hold), dt);
    out[slot_d] = L.a0 + L.a1 * te.t + L.a2 * te.t2 + L.a3 * te.t3 + L.a4 * te.t4 + L.a5 * te.t5;     // fp.py:688, :719
  }
}

// The NaN rule of the box prepass below for one step (a NaN x or y): fot_assess, which reads every step of a trajectory
// itself, applies it with this function.  The prepass keeps its expression written out: calling this function there
// changes the instructions ptxas schedules for fot_prepass.
__device__ __forceinline__ bool nan_step(double2 o) { return (o.x != o.x) || (o.y != o.y); }

// Boxes of the predicted trajectories, once per launch: one warp per trajectory (q, sample, ped),
// (xmin, xmax, ymin, ymax) over all its steps rounded outward to fp32.  A NaN anywhere makes the
// whole box NaN, which fails every overlap test: exactly the reference's prefilter, whose np.min /
// np.max propagate the NaN and thereby remove that pedestrian from the test (fp.py:1211-1222).
constexpr int kBoxPerWarp = 4;   // trajectories boxed per warp of fot_prepass: their loads are all in flight together
__device__ __forceinline__ void aabb_prepass_body(const double2* __restrict__ dyn, float4* __restrict__ box, long long n_traj, int T_obs,
                                                  unsigned block) {
  const long long warp = ((long long)block * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const long long t0 = warp * kBoxPerWarp;
  if (t0 >= n_traj) return;
  // both loads of each of the warp's <= 64-step trajectories are issued before the first comparison
  const bool h0 = lane < T_obs, h1 = lane + 32 < T_obs;
  double2 o0[kBoxPerWarp], o1[kBoxPerWarp];
#pragma unroll
  for (int u = 0; u < kBoxPerWarp; ++u) {
    const double2* src = dyn + (size_t)min(t0 + u, n_traj - 1) * T_obs;
    o0[u] = h0 ? src[lane] : make_double2(INFINITY, INFINITY);
    o1[u] = h1 ? src[lane + 32] : o0[u];
  }
#pragma unroll
  for (int u = 0; u < kBoxPerWarp; ++u) {
    if (t0 + u >= n_traj) break;
    const double2* src = dyn + (size_t)(t0 + u) * T_obs;
    bool bad = (h0 && ((o0[u].x != o0[u].x) || (o0[u].y != o0[u].y))) || (h1 && ((o1[u].x != o1[u].x) || (o1[u].y != o1[u].y)));
    double xlo = h0 ? fmin(o0[u].x, o1[u].x) : INFINITY, xhi = h0 ? fmax(o0[u].x, o1[u].x) : -INFINITY;
    double ylo = h0 ? fmin(o0[u].y, o1[u].y) : INFINITY, yhi = h0 ? fmax(o0[u].y, o1[u].y) : -INFINITY;
    for (int k = lane + 64; k < T_obs; k += 32) {
      const double2 o = src[k];
      bad |= (o.x != o.x) || (o.y != o.y);
      xlo = fmin(xlo, o.x); xhi = fmax(xhi, o.x); ylo = fmin(ylo, o.y); yhi = fmax(yhi, o.y);
    }
    // outward rounding to fp32 is monotone, so it commutes with min / max: round first, then reduce the ordered-uint
    // images with one redux each (four instructions instead of forty shuffles and as many fp64 comparisons)
    const unsigned rxlo = __reduce_min_sync(0xffffffffu, f2ord(__double2float_rd(xlo)));
    const unsigned rxhi = __reduce_max_sync(0xffffffffu, f2ord(__double2float_ru(xhi)));
    const unsigned rylo = __reduce_min_sync(0xffffffffu, f2ord(__double2float_rd(ylo)));
    const unsigned ryhi = __reduce_max_sync(0xffffffffu, f2ord(__double2float_ru(yhi)));
    bad = __any_sync(0xffffffffu, bad);
    if (lane == 0) {
      const float nanf_ = __int_as_float(0x7fc00000);
      box[t0 + u] = bad ? make_float4(nanf_, nanf_, nanf_, nanf_) : make_float4(ord2f(rxlo), ord2f(rxhi), ord2f(rylo), ord2f(ryhi));
    }
  }
}

// One launch for both prepasses (they are independent and each too small to fill the GPU for long):
// blocks [0, n_cost_blocks) build the cost tables, the rest box the predicted trajectories.  (Spreading the two kinds
// evenly over the grid, so that every SM runs FP64-bound and memory-bound blocks together, measured slower: 0.142 against
// 0.133 ms.)
__global__ void __launch_bounds__(256)
fot_prepass(const Plan P, const Batch B, double* __restrict__ cost_tab, unsigned n_cost_blocks,
            const double2* __restrict__ dyn, float4* __restrict__ box, long long n_traj, int T_obs) {
  if (blockIdx.x < n_cost_blocks) cost_prepass_body(P, B, cost_tab, blockIdx.x);
  else aabb_prepass_body(dyn, box, n_traj, T_obs, blockIdx.x - n_cost_blocks);
}

// ----------------------------------------------------------------------------------------
// Regeneration of one candidate by a whole block, in the reference's arithmetic order: decode the generation-order
// index i of query q (fp.py:398-449, brake ladder appended), solve its two profiles, convert every sample to Cartesian.
// W (and MW, when not null) receive the [FOT_N_SERIES][NT] rows, samples [0, N); kStore false: nothing is stored, only
// the length is found.  `tt` is the block's [NT][kTT] time table; *s_first_nan must hold 0x7fffffff and be visible to the
// block on entry.  Returns to every thread the samples kept after the NaN-prefix truncation (first NaN x, else N).
// ----------------------------------------------------------------------------------------
template <bool kStore = true>
__device__ __forceinline__ int regenerate(const Plan& P, const Batch& B, int q, int i, const double* tt, double* W,
                                          double* MW, int* s_first_nan) {
  const int NT = P.n_t_max, tid = threadIdx.x;
  const double* fs = B.frenet + 6 * (size_t)q;
  const int n_v = B.n_v[q], n_d = P.cfg.n_d;
  const int grid_total = P.cfg.n_T * n_v * n_d;
  Lon lon;
  Lat lat;
  int N;
  if (i < grid_total) {
    const int id = i % n_d, kv = (i / n_d) % n_v, jT = i / (n_d * n_v);
    N = P.n_steps[jT] + 1;
    lon = lon_solve(fs, B.v_grid[(size_t)q * B.n_v_max + kv], P.T[jT], P.inv4 + 4 * jT, n_v == 1, N - 1);
    lat = lat_solve(fs, P.d_grid[id], P.T[jT], P.inv5 + 9 * jT, n_d == 1, N - 1);
  } else {
    const int bi = i - grid_total;
    N = P.cfg.n_total;
    lon = lon_solve(fs, 0.0, P.Tb[bi], P.inv4b + 4 * bi, true, P.n_steps_b[bi]);
    lat = lat_solve(fs, fs[3], P.Tb[bi], P.inv5b + 9 * bi, true, P.n_steps_b[bi]);
  }
  for (int n = tid; n < N; n += blockDim.x) {
    const double s = lon_p0(lon, tt, n), sd = lon_p1(lon, tt, n), sdd = lon_p2(lon, tt, n);
    const double d = lat_p0(lat, tt, n), dd = lat_p1(lat, tt, n), ddd = lat_p2(lat, tt, n);
    const RefPt r = spline_ref(P, s);
    double sn, cs;
    sincos(r.rth, &sn, &cs);
    const CartPt cp = to_cartesian(r.rx, r.ry, cs, sn, r.rth, r.rk, r.rdk, sd, sdd, d, dd, ddd);
    if (cp.x != cp.x) atomicMin(s_first_nan, n);
    if (!kStore) continue;
    W[0 * NT + n] = tt[kTT * n];
    W[1 * NT + n] = s;   W[2 * NT + n] = sd;  W[3 * NT + n] = sdd; W[4 * NT + n] = lon_p3(lon, tt, n);
    W[5 * NT + n] = d;   W[6 * NT + n] = dd;  W[7 * NT + n] = ddd; W[8 * NT + n] = lat_p3(lat, tt, n);
    W[9 * NT + n] = cp.x; W[10 * NT + n] = cp.y; W[11 * NT + n] = wrap_angle(cp.ang);
    W[12 * NT + n] = cp.kappa; W[13 * NT + n] = cp.v; W[14 * NT + n] = cp.a;
    if (MW) {
      // the same values into the mirror: plain stores, which the memory system carries over NVLink when the mirror is
      // a peer's memory -- the gather of the sharded sweep happens here, without a collective call
#pragma unroll
      for (int r = 0; r < FOT_N_SERIES; ++r) MW[r * NT + n] = W[r * NT + n];
    }
  }
  __syncthreads();
  return *s_first_nan < N ? *s_first_nan : N;
}

// ----------------------------------------------------------------------------------------
// Winner kernel: one block per query.
// ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
fot_winner(const Plan P, const Batch B, const Out O, int parts_per_query) {
  extern __shared__ double sm[];
  const int NT = P.n_t_max;
  double* tt = sm;   // [NT][kTT]
  __shared__ double s_cost[4];
  __shared__ int s_idx[4];
  __shared__ int s_first_nan;
  const int q = blockIdx.x, tid = threadIdx.x;

  double c = INFINITY;
  int i = 0x7fffffff;
  for (int p = tid; p < parts_per_query; p += blockDim.x) {
    const int pi = O.part_idx[(size_t)q * parts_per_query + p];
    if (pi >= 0) argmin_merge(c, i, O.part_cost[(size_t)q * parts_per_query + p], pi);
  }
  for (int off = 16; off > 0; off >>= 1) {
    const double oc = __shfl_down_sync(0xffffffffu, c, off);
    const int oi = __shfl_down_sync(0xffffffffu, i, off);
    argmin_merge(c, i, oc, oi);
  }
  if ((tid & 31) == 0) { s_cost[tid >> 5] = c; s_idx[tid >> 5] = i; }
  if (tid == 0) s_first_nan = 0x7fffffff;
  for (int n = tid; n < NT; n += blockDim.x) tt_fill(tt, n, P.cfg.dt);
  __syncthreads();
  c = s_cost[0]; i = s_idx[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) argmin_merge(c, i, s_cost[w], s_idx[w]);
  double* W = O.winner + (size_t)q * FOT_N_SERIES * NT;
  double* MW = O.m_winner ? O.m_winner + (size_t)q * FOT_N_SERIES * NT : nullptr;       // mirror (peer memory), see Out
  if (O.m_stats && tid < FOT_N_STATS) O.m_stats[(size_t)q * FOT_N_STATS + tid] = O.stats[(size_t)q * FOT_N_STATS + tid];   // final since the sweep
  Plan V;                                                // the query's route (the sweep left no partial for a bad id)
  if (!route_plan(P, B.rt, q, V)) i = 0x7fffffff;
  if (i == 0x7fffffff) {
    if (tid == 0) {
      O.best_idx[q] = -1; O.best_cost[q] = INFINITY; O.winner_len[q] = 0;
      if (O.m_best_idx) { O.m_best_idx[q] = -1; O.m_best_cost[q] = INFINITY; O.m_winner_len[q] = 0; }
    }
    return;
  }
  const int len = regenerate(V, B, q, i, tt, W, MW, &s_first_nan);
  if (tid == 0) {
    O.best_idx[q] = i;
    O.best_cost[q] = c;
    O.winner_len[q] = len;
    if (O.m_best_idx) { O.m_best_idx[q] = i; O.m_best_cost[q] = c; O.m_winner_len[q] = len; }
  }
}

// One word per rank in the gather root's memory: the sequence number of the last step whose winner block is complete
// there.  Launched behind fot_winner in stream order; the fence makes the mirror stores visible system-wide first.
__global__ void fot_publish_kernel(unsigned* flag, unsigned seq) {
  __threadfence_system();
  *reinterpret_cast<volatile unsigned*>(flag) = seq;
}
// Root side: wait (bounded) until every rank has published `seq` or later.  err: set to 1 on time-out.
__global__ void fot_await_kernel(const unsigned* flags, int world, unsigned seq, long long timeout_ns, unsigned* err) {
  const int r = threadIdx.x;
  if (r >= world) return;
  long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (;;) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + r) : "memory");
    if ((int)(v - seq) >= 0) break;
    long long now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
    if (now - t0 > timeout_ns) { *err = 1u; break; }
    __nanosleep(200);
  }
}

// ----------------------------------------------------------------------------------------
// FMA pipe probes (roofline denominators).  8 independent chains per thread.
// ----------------------------------------------------------------------------------------
template <int KIND>
__global__ void fot_probe_kernel(float* sink, int iters) {
  if (KIND == 0) {
    double a[8];
    for (int i = 0; i < 8; ++i) a[i] = 1.0 + 1e-9 * (threadIdx.x + i);
    const double m = 1.0000001, c = 1e-7;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = fma(a[i], m, c);
    }
    double s = 0;
    for (int i = 0; i < 8; ++i) s += a[i];
    if (s == 12345.678) sink[0] = (float)s;
  } else if (KIND == 1) {
    float a[8];
    for (int i = 0; i < 8; ++i) a[i] = 1.0f + 1e-6f * (threadIdx.x + i);
    const float m = 1.000001f, c = 1e-6f;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = fmaf(a[i], m, c);
    }
    float s = 0;
    for (int i = 0; i < 8; ++i) s += a[i];
    if (s == 12345.678f) sink[0] = s;
  } else {
    unsigned long long a[8];
    for (int i = 0; i < 8; ++i) {
      const float lo = 1.0f + 1e-6f * (threadIdx.x + i), hi = 1.0f + 2e-6f * (threadIdx.x + i);
      a[i] = ((unsigned long long)__float_as_uint(hi) << 32) | __float_as_uint(lo);
    }
    const float mf = 1.000001f, cf = 1e-6f;
    const unsigned long long m = ((unsigned long long)__float_as_uint(mf) << 32) | __float_as_uint(mf);
    const unsigned long long c = ((unsigned long long)__float_as_uint(cf) << 32) | __float_as_uint(cf);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int i = 0; i < 8; ++i)
          asm volatile("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(a[i]) : "l"(m), "l"(c));
    }
    unsigned long long s = 0;
    for (int i = 0; i < 8; ++i) s ^= a[i];
    if (s == 0x123456789abcdefULL) sink[0] = 1.0f;
  }
}

}  // namespace fot
