// fot_sweep_items.cuh -- the sample-major sweep kernel (sm_100a, fp64).
//
// One fused kernel for the whole candidate sweep of every query, per-CTA arg-min partials out (reduced
// by fot_winner, fot_kernels.cuh), no trajectory written to HBM.  The work is laid out sample-major:
//
//   block  = (query, horizon T_j, chunk of terminal speeds)  -- or the query's brake ladder;
//            a CTA sweeps `bpc` consecutive blocks of one query (all of them in large batches), so
//            the obstacle staging, the spline tables and the arg-min / histogram are per CTA
//   thread = one (terminal speed v_k, sample t_n) "item": everything that depends on the
//            longitudinal profile only -- s(t_n), the spline reference point, heading, curvature,
//            1/s_dot -- is computed ONCE per item and lives in registers;
//   loop   = the lateral targets d_i.  The quintic solve is linear in the target, so at a fixed
//            sample  d_i(t_n) = A + d_i * B, and with it every first-order quantity of the
//            Frenet->Cartesian map (q = 1 - kappa_r d, d', d'', kappa_r' d + kappa_r d', the step
//            vector to the previous sample) is AFFINE in d_i: one FMA each from per-thread constants.
//            The limit checks are evaluated in squared, division-free form
//              kappa = w / h^3,  a = Z / (h q),  v^2 = s_dot^2 h^2   (h^2 = q^2 + d'^2)
//              |kappa| > k_max  <=>  w^2 > k_max^2 h^6       (no sqrt, no reciprocal, no atan2)
//            so the inner loop is ~45 FP64 instructions per candidate sample.
//
// A candidate's validity flags (priority chain fp.py:964-991, silent drops :933-956) are an OR over
// its samples, i.e. over the threads of one speed: warp `redux.or` over the lanes of that speed,
// then one shared-memory atomic per 4 candidates.  The NaN-prefix truncation (fp.py:851-875) depends
// on the reference point only, so it is a per-speed constant, not per-candidate state.
//
// Collision (fp.py:1035-1233): a clean candidate's sample lies exactly on the normal of the
// reference line through the item's reference point at lateral offset |d| <= road half-width, so an
// obstacle sample can only touch it when it is within r along the tangent and W + r across it.
//   1. fot_aabb_prepass (one warp per predicted trajectory) boxes every trajectory once per launch;
//      a block keeps only the trajectories whose box meets the box of its own reference points --
//      the reference's own AABB prefilter (fp.py:1211-1222) including its NaN-trajectory rule;
//   2. each item tests the listed obstacles at its own time step against the tangent-frame window
//      (the obstacle tensor is read in the reference's [S][P][T][2] layout: consecutive lanes are
//      consecutive time steps, so the 16-byte loads coalesce; small fields are staged in shared memory
//      by ONE bulk copy, cp.async.bulk + mbarrier) and remembers the few survivors in a bit mask;
//   3. survivors go to a block-wide queue that all threads drain, one entry each, with the exact
//      `dx*dx + dy*dy <= r^2` against every still-alive clean candidate of that speed.
//
// Numerics: costs are bit-identical to the reference (same arithmetic order, NumPy pairwise
// sums); the validity chain uses algebraically equal forms that differ by a few ulp (see
// DESIGN.md section 7); the winner's sequences are regenerated in reference order by fot_winner.
// The squared forms assume non-negative limits (a negative limit rejects everything, as in the
// reference).
//
// The upload gate, the boxes of a staged obstacle block, the reference point and the flag idiom are shared with
// fot_sweep_pairs (fot_sweep_math.cuh); the cost tables and trajectory boxes come from fot_prepass (fot_kernels.cuh).
#pragma once
#include <type_traits>
#include "fot_sweep_math.cuh"

namespace fot {

// Optional phase timeline (tuning only): -DFOT_PHASE_CLOCKS accumulates, per warp, the clock64 span
// between the kernel's barriers into g_phase_clk[phase] (read back with fot_debug_phase_clocks).
#ifdef FOT_PHASE_CLOCKS
__device__ unsigned long long g_phase_clk[16];
#define FOT_PHASE_MARK(k) do { const long long t__ = clock64(); if (lane == 0) atomicAdd(&g_phase_clk[k], (unsigned long long)(t__ - t_phase)); t_phase = t__; } while (0)
#else
#define FOT_PHASE_MARK(k) do { } while (0)
#endif

#ifndef FOT_ITEM_MIN_CTAS
#define FOT_ITEM_MIN_CTAS 2
#endif
constexpr int kItemThreads = 320;   // largest block of fot_sweep_items

struct ItemGeom {
  int32_t ppc;               // terminal speeds (pairs) per grid block
  int32_t chunks;            // grid blocks per horizon
  int32_t grid_blocks;       // n_T * chunks
  int32_t ppb;               // brake horizons per brake block
  int32_t brake_blocks;
  int32_t blocks_per_query;
  int32_t bpc;               // blocks swept by one CTA (consecutive blocks of one query)
  int32_t ctas_per_query;    // ceil(blocks_per_query / bpc)
  int32_t threads;           // block size (multiple of 32, >= items of the largest block)
  int32_t pcap;              // max(ppc, ppb): per-pair table slots
  int32_t ct_lcap;           // max(n_d, ppb): lateral slots of the staged cost-table entries
  int32_t qcap;              // collision queue capacity (entries)
  int32_t ochunk;            // list entries culled per queue round
  int32_t lcap;              // obstacle list capacity (static + dynamic entries)
  int32_t stage_dyn;         // 1: the query's obstacle block is staged in shared memory by one bulk copy
  int32_t spline_smem;       // 1: spline tables copied to shared memory
  int32_t vwords;            // u32 words per candidate of the chance-constraint violation bitmap (0: no budget)
  int32_t nw4, nwc;          // flag words (4 candidates each) / bit-mask words (32 candidates each) per pair
  int32_t n_zero;            // u32 words of the zero-initialised region starting at o_flags
  // byte offsets into dynamic shared memory
  int32_t o_row, o_sdl, o_ct, o_dgrid, o_vlast, o_spl, o_dyn;
  int32_t o_fn, o_flags, o_hit, o_viol, o_queue, o_list, o_slow, o_clean;
  // gated launch (host-pointer call): the sweep is launched before / while the obstacle tensor is uploaded in
  // slices of gate_per queries; the upload streams set gate[slice] = gate_epoch behind each slice and a CTA waits
  // for the slice of its own query.  With fused_box the trajectory boxes are computed by the CTA from its staged obstacle
  // block (no prepass over a tensor that has not arrived yet).
  int32_t fused_box;         // 1: boxes from the staged block into shared memory at o_box (needs stage_dyn)
  int32_t o_box;
  int32_t gate_q0;           // index of this launch's first query in the uploaded batch
  int32_t gate_per;          // queries per upload slice
  uint32_t gate_epoch;
  unsigned* gate;            // [slice] flags, [kGateSlices] set to 1 by a CTA that gave up waiting; nullptr: no gate
};

// The spline tables in shared memory (spline_smem) or the Plan's own arrays.
struct SplineView {
  const double *knots, *xa, *xb, *xc, *xd, *ya, *yb, *yc, *yd;
  int nx;
};
// spline_ref_tab over the tables of a SplineView.
struct SplineViewTab {
  const SplineView& V;
  __device__ __forceinline__ double operator()(int k, int i) const {
    const double* t[9] = {V.knots, V.xa, V.xb, V.xc, V.xd, V.ya, V.yb, V.yc, V.yd};
    return t[k][i];
  }
};

// Bit i of the result: candidate 32*w + i of pair `pp` has no validity flag (4 flag bytes per word).
__device__ __forceinline__ unsigned clean_word(const unsigned* flags_pp, int nw4, int n_dl, int w) {
  unsigned m = 0u;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int w4 = 8 * w + k;
    if (w4 < nw4) {
      const unsigned x = flags_pp[w4];
      const unsigned t = ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;   // bit 7 of every zero byte
      m |= ((((t >> 7) * 0x00204081u) >> 21) & 0xfu) << (4 * k);
    }
  }
  const int rem = n_dl - 32 * w;
  return rem >= 32 ? m : (m & ((1u << rem) - 1u));
}

// kFused: the variant of the gated host-pointer call (waits for its query's upload slice, boxes the trajectories
// itself).  kRoutes: every query on its own reference path (Batch::rt, DESIGN.md section 4h).  Template parameters
// rather than run-time branches: the resident path keeps exactly the code (and the register allocation) it is tuned for.
template <bool kFused, bool kRoutes = false>
__global__ void __launch_bounds__(kItemThreads, FOT_ITEM_MIN_CTAS)
fot_sweep_items(const Plan P, const Batch B, const Out O, const ItemGeom G) {
  extern __shared__ __align__(16) unsigned char smb[];
  double* row = reinterpret_cast<double*>(smb + G.o_row);      // [pcap][NT][kRowW]
  double* sdl = reinterpret_cast<double*>(smb + G.o_sdl);      // [pcap] s_dot at the last sample
  double* ctb = reinterpret_cast<double*>(smb + G.o_ct);       // [pcap + 2 max(n_d, ppb)] this block's cost-table entries: Js | Jp | d_end
  double* dgrid = reinterpret_cast<double*>(smb + G.o_dgrid);  // [n_d]
  double* vlast = reinterpret_cast<double*>(smb + G.o_vlast);  // [pcap][n_d]  v^2 at the last kept sample
  double* spl = reinterpret_cast<double*>(smb + G.o_spl);      // [9][nx] when spline_smem
  const double2* dynst = reinterpret_cast<const double2*>(smb + G.o_dyn);   // [SP][T_obs] when stage_dyn
  int* pi_fn = reinterpret_cast<int*>(smb + G.o_fn);                // [pcap] first NaN sample (INT_MAX: none)
  unsigned* flags = reinterpret_cast<unsigned*>(smb + G.o_flags);   // [pcap][nw4]
  unsigned* hitw = reinterpret_cast<unsigned*>(smb + G.o_hit);      // [pcap][nwc] decisive collision
  unsigned* viol = reinterpret_cast<unsigned*>(smb + G.o_viol);     // [pcap][n_d][vwords]
  unsigned* queue = reinterpret_cast<unsigned*>(smb + G.o_queue);   // [qcap]
  unsigned* olist = reinterpret_cast<unsigned*>(smb + G.o_list);   // [lcap] element offsets: static j (first M slots), dynamic j * T_obs
  unsigned* cleanw = reinterpret_cast<unsigned*>(smb + G.o_clean);  // [pcap][nwc] kinematically clean (phase D)
  unsigned short* slowq = reinterpret_cast<unsigned short*>(smb + G.o_slow);   // [threads] items with a low-speed sample
  __shared__ int s_qcount[2];
  __shared__ int s_next[2];             // work counters of the collision rounds
  __shared__ int s_nlist[2];            // static / dynamic list lengths
  __shared__ int s_nslow;               // items in the low-speed queue
  __shared__ unsigned s_box[4];         // xmin xmax ymin ymax of the block's reference points (ordered-uint floats)
  __shared__ int s_stats[FOT_N_STATS];
  __shared__ double s_cost[kItemThreads / 32];
  __shared__ int s_idx[kItemThreads / 32];
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ int s_abort;
  float4* sbox = reinterpret_cast<float4*>(smb + G.o_box);          // [SP] trajectory boxes when fused_box

  const int NT = P.n_t_max;
  const int q = blockIdx.x / G.ctas_per_query;
  const int cta = blockIdx.x - q * G.ctas_per_query;
  const int tid = threadIdx.x, lane = tid & 31, bd = blockDim.x;
  const double* fs = B.frenet + 6 * (size_t)q;
  const int n_v = B.n_v[q];
  const int n_d = P.cfg.n_d;
  const double dt = P.cfg.dt;
  const size_t part = (size_t)q * G.ctas_per_query + cta;
  const int b_first = cta * G.bpc, b_last = min(G.blocks_per_query, b_first + G.bpc);
  // A non-finite Frenet state makes every sample of every candidate non-finite: the reference drops
  // them all silently (empty / non-finite guards fp.py:933-946).
  const bool state_ok = fabs(fs[0]) + fabs(fs[1]) + fabs(fs[2]) + fabs(fs[3]) + fabs(fs[4]) + fabs(fs[5]) < INFINITY;

  const bool has_dyn = B.dyn_raw != nullptr;
  const int SP = has_dyn ? B.S * B.P : 0;
  const int M = B.static_raw ? B.n_static : 0;
  const double2* dyn_q = has_dyn ? reinterpret_cast<const double2*>(B.dyn_raw) + (size_t)q * SP * B.T_obs : nullptr;
  const double2* stat_q = M > 0 ? reinterpret_cast<const double2*>(B.static_raw) + (size_t)(B.static_per_query ? q : 0) * M : nullptr;

  // ---- once per CTA: obstacle block in flight, grids and spline tables in shared memory ----------
  Plan PR_;                                               // kRoutes: the query's route (route_plan, below)
  const Plan& PS = kRoutes ? PR_ : P;                    // spline tables and knot count of this query
  if (kFused && G.gate && gate_wait(G, q, s_abort)) return;
  if (tid == 0 && G.stage_dyn && state_ok) {
    mbar_init(&s_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const uint32_t bytes = (uint32_t)SP * (uint32_t)B.T_obs * 16u;
    mbar_expect_tx(&s_bar, bytes);
    tma_bulk_g2s(smb + G.o_dyn, dyn_q, bytes, &s_bar);
  }
  if (tid < FOT_N_STATS) s_stats[tid] = 0;
  for (int i = tid; i < n_d; i += bd) dgrid[i] = P.d_grid[i];
  if constexpr (kRoutes) {
    // the route's id is read behind the bulk copy; a bad id plans nothing (the copy must have landed before the CTA
    // exits; thread 0 initialised the barrier and waits on it)
    if (!route_plan(P, B.rt, q, PR_)) {
      if (tid == 0) {
        if (G.stage_dyn && state_ok) mbar_wait(&s_bar, 0u);
        O.part_cost[part] = INFINITY; O.part_idx[part] = -1;
      }
      return;
    }
  }
  if (G.spline_smem) {
    const int nx = PS.cfg.nx;
    for (int i = tid; i < nx; i += bd) {
      spl[i] = PS.knots[i];
      spl[nx + i] = PS.xa[i];      spl[3 * nx + i] = PS.xc[i];
      spl[5 * nx + i] = PS.ya[i];  spl[7 * nx + i] = PS.yc[i];
      if (i < nx - 1) {
        spl[2 * nx + i] = PS.xb[i]; spl[4 * nx + i] = PS.xd[i];
        spl[6 * nx + i] = PS.yb[i]; spl[8 * nx + i] = PS.yd[i];
      }
    }
  }
  double my_cost = INFINITY;            // running arg-min over every block this CTA sweeps
  int my_idx = 0x7fffffff;
  bool boxes_done = false;
#ifdef FOT_PHASE_CLOCKS
  long long t_phase = clock64();
#endif

  for (int b = b_first; b < b_last; ++b) {
  const bool brake_blk = b >= G.grid_blocks;
  // ---- which pairs does this block own? -----------------------------------------------------
  int jT = 0, k_lo = 0, n_k = 0, N = 0, n_dl = 0;
  if (!brake_blk) {
    jT = b / G.chunks;
    k_lo = (b - jT * G.chunks) * G.ppc;
    n_k = min(G.ppc, n_v - k_lo);
    N = P.n_steps[jT] + 1;
    n_dl = n_d;
  } else {
    const int b0 = (b - G.grid_blocks) * G.ppb;
    if (fs[1] > 0.1 && b0 < P.cfg.n_B) {                 // fp.py:469 BRAKE_MIN_SPEED
      k_lo = b0;
      n_k = min(G.ppb, P.cfg.n_B - b0);
    }
    N = P.cfg.n_total;
    n_dl = 1;
  }
  if (n_k <= 0) continue;                                // uniform per block
  const int n_cand = n_k * n_dl;
  const int cand0 = brake_blk ? P.cfg.n_T * n_v * n_d + k_lo : (jT * n_v + k_lo) * n_d;   // generation order (fp.py:398-449)
  if (!state_ok) {
    for (int c = tid; c < n_cand; c += bd) {
      if (O.cand_cat) O.cand_cat[(size_t)q * O.cand_stride + cand0 + c] = (uint8_t)FOT_CAT_DROP;
      if (O.cand_cost) O.cand_cost[(size_t)q * O.cand_stride + cand0 + c] = qnan();
    }
    continue;
  }

  // ---- phase A: per-block shared-memory state ------------------------------------------------------
  if (tid == 0) {
    s_qcount[0] = 0; s_qcount[1] = 0; s_next[0] = 0; s_next[1] = 0; s_nlist[0] = 0; s_nlist[1] = 0; s_nslow = 0;
    s_box[0] = 0xffffffffu; s_box[1] = 0u; s_box[2] = 0xffffffffu; s_box[3] = 0u;
  }
  if (tid < G.pcap) pi_fn[tid] = 0x7fffffff;
  for (int i = tid; i < G.n_zero; i += bd) flags[i] = 0u;          // flags | hit words | violation bitmaps
  {
    // this block's jerk sums / terminal offsets (fot_prepass tables) -> shared memory, asynchronously:
    // phase E reads them four barriers from now
    const int nTv = P.cfg.n_T * B.n_v_max, nTd = P.cfg.n_T * n_d, nB = P.cfg.n_B;
    const double* ct = B.cost_tab + (size_t)q * (nTv + 2 * nTd + 3 * nB);
    const int n_lat = brake_blk ? n_k : n_d, lcap = G.ct_lcap;
    if (tid < n_k + 2 * n_lat) {
      const double* src;
      double* dst;
      if (tid < n_k) {
        src = brake_blk ? ct + nTv + 2 * nTd + k_lo + tid : ct + jT * B.n_v_max + k_lo + tid;
        dst = ctb + tid;
      } else if (tid < n_k + n_lat) {
        const int li = tid - n_k;
        src = brake_blk ? ct + nTv + 2 * nTd + nB + k_lo + li : ct + nTv + jT * n_d + li;
        dst = ctb + G.pcap + li;
      } else {
        const int li = tid - n_k - n_lat;
        src = brake_blk ? ct + nTv + 2 * nTd + 2 * nB + k_lo + li : ct + nTv + nTd + jT * n_d + li;
        dst = ctb + G.pcap + lcap + li;
      }
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  FOT_PHASE_MARK(0);
  __syncthreads();
  FOT_PHASE_MARK(1);

  // ---- phase B: one item per thread ---------------------------------------------------------------
  const int n_items = n_k * N;
  const bool active = tid < n_items;
  const int p = active ? tid / N : -1;                                         // pair slot of this item
  const int n = active ? tid - p * N : 0;                                      // its sample
  double i_rx = 0, i_ry = 0, i_cth = 0, i_sth = 0, i_rk = 0, i_rdk = 0, i_sd = 0, i_sdd = 0, i_isd = 0;
  double A0 = 0, B0 = 0, A1 = 0, B1 = 0, A2 = 0, B2 = 0;
  if (active) {
    // quartic solve of the item's own pair (fp.py:619-647) -- a dozen flops, cheaper than a barrier
    Lon L;
    if (!brake_blk)
      L = lon_solve(fs, B.v_grid[(size_t)q * B.n_v_max + k_lo + p], P.T[jT], P.inv4 + 4 * jT, n_v == 1, N - 1);
    else
      L = lon_solve(fs, 0.0, P.Tb[k_lo + p], P.inv4b + 4 * (k_lo + p), true, P.n_steps_b[k_lo + p]);
    const bool held = n > L.hold;                                              // fp.py:487-499 brake padding
    const TPow tp = tpow(held ? L.hold : n, dt);
    const double s = L.a0 + L.a1 * tp.t + L.a2 * tp.t2 + L.a3 * tp.t3 + L.a4 * tp.t4;             // fp.py:644
    i_sd = held ? 0.0 : L.a1 + 2.0 * L.a2 * tp.t + 3.0 * L.a3 * tp.t2 + 4.0 * L.a4 * tp.t3;      // fp.py:645
    i_sdd = held ? 0.0 : 2.0 * L.a2 + 6.0 * L.a3 * tp.t + 12.0 * L.a4 * tp.t2;                    // fp.py:646
    SplineView V;
    V.nx = PS.cfg.nx;
    if (G.spline_smem) {
      const int nx = V.nx;
      V.knots = spl; V.xa = spl + nx; V.xb = spl + 2 * nx; V.xc = spl + 3 * nx; V.xd = spl + 4 * nx;
      V.ya = spl + 5 * nx; V.yb = spl + 6 * nx; V.yc = spl + 7 * nx; V.yd = spl + 8 * nx;
    } else {
      V.knots = PS.knots; V.xa = PS.xa; V.xb = PS.xb; V.xc = PS.xc; V.xd = PS.xd;
      V.ya = PS.ya; V.yb = PS.yb; V.yc = PS.yc; V.yd = PS.yd;
    }
    const RefFast rp = spline_ref_tab(SplineViewTab{V}, V.nx, s);
    i_rx = rp.rx; i_ry = rp.ry; i_cth = rp.cth; i_sth = rp.sth; i_rk = rp.rk; i_rdk = rp.rdk;
    i_isd = fabs(i_sd) > 1e-3 ? rcp_nr(i_sd) : 0.0;                            // fp.py:792 EPS_S_DOT
    // lateral basis at this sample: d_i(t) = A(t) + d_i * B(t) (the quintic's right-hand side is linear
    // in the target, fp.py:676-683); Horner with running derivatives
    double c0, c1, c2, c3, c4, c5, b3, b4, b5;
    if (!brake_blk) {
      const double T = P.T[jT];
      const double* Ai = P.inv5 + 9 * jT;
      c0 = fs[3]; c1 = fs[4]; c2 = fs[5] / 2.0;
      const double r0 = -c0 - c1 * T - c2 * T * T, r1 = -c1 - 2.0 * c2 * T, r2 = -2.0 * c2;
      c3 = fma(r2, Ai[2], fma(r1, Ai[1], r0 * Ai[0]));
      c4 = fma(r2, Ai[5], fma(r1, Ai[4], r0 * Ai[3]));
      c5 = fma(r2, Ai[8], fma(r1, Ai[7], r0 * Ai[6]));
      b3 = Ai[0]; b4 = Ai[3]; b5 = Ai[6];
    } else {                                                                   // one lateral profile per brake horizon (fp.py:480-482)
      const Lat Lb = lat_solve(fs, fs[3], P.Tb[k_lo + p], P.inv5b + 9 * (k_lo + p), true, P.n_steps_b[k_lo + p]);
      c0 = Lb.a0; c1 = Lb.a1; c2 = Lb.a2; c3 = Lb.a3; c4 = Lb.a4; c5 = Lb.a5;
      b3 = b4 = b5 = 0.0;
    }
    {
      const double t = tp.t;
      double pA = fma(c5, t, c4), dA = c5, ddA;
      ddA = dA;               dA = fma(dA, t, pA);  pA = fma(pA, t, c3);
      ddA = fma(ddA, t, dA);  dA = fma(dA, t, pA);  pA = fma(pA, t, c2);
      ddA = fma(ddA, t, dA);  dA = fma(dA, t, pA);  pA = fma(pA, t, c1);
      ddA = fma(ddA, t, dA);  dA = fma(dA, t, pA);  pA = fma(pA, t, c0);
      double pB = fma(b5, t, b4), dB = b5, ddB;
      ddB = dB;               dB = fma(dB, t, pB);  pB = fma(pB, t, b3);
      ddB = fma(ddB, t, dB);  dB = fma(dB, t, pB);  pB = pB * t;
      ddB = fma(ddB, t, dB);  dB = fma(dB, t, pB);  pB = pB * t;
      ddB = fma(ddB, t, dB);  dB = fma(dB, t, pB);  pB = pB * t;
      A0 = pA; B0 = pB;
      A1 = held ? 0.0 : dA;        B1 = held ? 0.0 : dB;
      A2 = held ? 0.0 : 2.0 * ddA; B2 = held ? 0.0 : 2.0 * ddB;
    }
    double* r = row + (p * NT + n) * kRowW;
    r[0] = i_rx; r[1] = i_ry; r[2] = i_cth; r[3] = i_sth; r[4] = i_rk; r[5] = s; r[6] = i_isd; r[7] = i_sd;
    r[8] = A0; r[9] = B0; r[10] = A1; r[11] = B1;
    if (i_rx != i_rx || i_ry != i_ry) atomicMin(&pi_fn[p], n);                 // fp.py:851-866
    if (n == N - 1) sdl[p] = i_sd;                                             // terminal speed of the cost (fp.py:724)
  }
  // box of the block's reference points (for the obstacle lists), fp32 rounded outward
  if (has_dyn || M > 0) {
    const bool ok = active && i_rx == i_rx && i_ry == i_ry;
    // ordered-uint encoding, warp min / max by redux, one atomic per warp and bound
    const unsigned xlo = __reduce_min_sync(0xffffffffu, ok ? f2ord(__double2float_rd(i_rx)) : 0xffffffffu);
    const unsigned xhi = __reduce_max_sync(0xffffffffu, ok ? f2ord(__double2float_ru(i_rx)) : 0u);
    const unsigned ylo = __reduce_min_sync(0xffffffffu, ok ? f2ord(__double2float_rd(i_ry)) : 0xffffffffu);
    const unsigned yhi = __reduce_max_sync(0xffffffffu, ok ? f2ord(__double2float_ru(i_ry)) : 0u);
    if (lane == 0 && xlo != 0xffffffffu) {
      atomicMin(&s_box[0], xlo); atomicMax(&s_box[1], xhi);
      atomicMin(&s_box[2], ylo); atomicMax(&s_box[3], yhi);
    }
  }
  FOT_PHASE_MARK(2);
  __syncthreads();
  FOT_PHASE_MARK(3);

  // ---- phase C: obstacle lists; validity chain, thread = item, loop = lateral targets -------------
  const int fn = active ? pi_fn[p] : 0;
  const int keep = fn == 0x7fffffff ? N : (fn >= 2 ? fn : 0);                  // fp.py:866
  const bool valid = active && n < keep;
  const bool chk = valid && n >= 1;                                            // limits skip index 0 (fp.py:964-983)
  const int n_circ = P.cfg.n_circles;
  double max_off = 0.0;                                  // footprint circles sit within max|offset| of the path point
  for (int i = 0; i < n_circ; ++i) max_off = fmax(max_off, fabs(P.cfg.circle_offsets[i]));
  const bool dist_mode = (B.dyn_mode == FOT_DYN_DISTRIBUTION);
  const double r2_dyn = dist_mode ? P.cfg.collide_r2 : P.cfg.collide_r2_single;   // fp.py:1099-1104, :1173
  const double rc_s = sqrt(P.cfg.collide_r2) * (1.0 + 1e-9) + 1e-9 + max_off;
  const double rc_d = sqrt(r2_dyn) * (1.0 + 1e-9) + 1e-9 + max_off;
  const double wroad = fmax(P.cfg.max_road_width + 1e-9, fabs(fs[3]));
  if (kFused && !boxes_done) {
    // first block of the CTA: box every predicted trajectory of the staged obstacle block
    mbar_wait(&s_bar, 0u);
    box_staged(dynst, sbox, SP, B.T_obs, tid >> 5, bd >> 5, lane);
    boxes_done = true;
    __syncthreads();
  }
  if (has_dyn || M > 0) {
    // keep the obstacles whose (trajectory) box meets the box of the reference points padded by the
    // widest reach of a clean candidate; a NaN box (fp.py:1211-1222) fails every comparison
    const float pad = __double2float_ru(wroad + fmax(rc_s, rc_d));
    const float bx0 = __fsub_rd(ord2f(s_box[0]), pad), bx1 = __fadd_ru(ord2f(s_box[1]), pad);
    const float by0 = __fsub_rd(ord2f(s_box[2]), pad), by1 = __fadd_ru(ord2f(s_box[3]), pad);
    if (s_box[0] != 0xffffffffu) {
      for (int j = tid; j < M; j += bd) {
        const double2 o = stat_q[j];
        if (o.x >= (double)bx0 && o.x <= (double)bx1 && o.y >= (double)by0 && o.y <= (double)by1) {
          const int slot = atomicAdd(&s_nlist[0], 1);
          olist[slot] = (unsigned)j;
        }
      }
      const float4* boxes = kFused ? sbox : B.dyn_box + (size_t)q * SP;
      for (int j = tid; j < SP; j += bd) {
        const float4 ob = boxes[j];                       // xmin xmax ymin ymax
        if (ob.x <= bx1 && ob.y >= bx0 && ob.z <= by1 && ob.w >= by0) {
          const int slot = atomicAdd(&s_nlist[1], 1);
          olist[M + slot] = (unsigned)(j * B.T_obs);
        }
      }
    }
  }
  const double* lim = B.limits + 4 * (size_t)q;
  const double inf = INFINITY;
  // squared limits; a negative limit rejects every checked sample, as `x > negative` does in the reference
  // (warp-uniform: pushed through redux so that they live in uniform registers, not in the 96 vector
  // registers the loop below is short of)
  auto uni = [&](double x) {
    const unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)__double2loint(x));
    const unsigned hi = __reduce_or_sync(0xffffffffu, (unsigned)__double2hiint(x));
    return __hiloint2double((int)hi, (int)lo);
  };
  const double vmax2 = uni(lim[0] < 0.0 ? -inf : lim[0] * lim[0]);
  const double amax2 = uni(lim[1] < 0.0 ? -inf : lim[1] * lim[1]);
  const double kmax2 = uni(lim[2] < 0.0 ? -inf : lim[2] * lim[2]);
  const double latmax2 = uni(lim[3] < 0.0 ? -inf : lim[3] * lim[3]);
  const double road_thr = P.cfg.max_road_width + 1e-9;                         // fp.py:982
  const double tele_thr = fmax(lim[0], P.cfg.max_speed) * dt * 3.0;            // fp.py:955
  const double tele2 = uni(tele_thr * tele_thr);
  const double fast2 = 0.25;                                                   // v > 0.5 (fp.py:1019)
  const unsigned keep4 = chk ? 0xffffffffu : F_DROP * 0x01010101u;             // n = 0: only the drop guards apply
  const double stop_dist = B.stop_dist[q];
  // per-item affine coefficients in d_i
  const double* rown = row + ((active ? p : 0) * NT + n) * kRowW;
  const double* rowp = chk ? rown - kRowW : rown;
  const double sd2 = i_sd * i_sd, isd2 = i_isd * i_isd;
  const double Q0 = fma(-i_rk, A0, 1.0), Q1 = -(i_rk * B0);                    // q = 1 - kappa_r d
  const double P0 = A1 * i_isd, P1 = B1 * i_isd;                               // d' (fp.py:792-799)
  const double R0 = (A2 - P0 * i_sdd) * isd2, R1 = (B2 - P1 * i_sdd) * isd2;   // d''
  const double M0 = fma(i_rdk, A0, i_rk * P0), M1 = fma(i_rdk, B0, i_rk * P1); // kappa_r' d + kappa_r d'
  const double S0 = i_sdd * Q0, S1 = i_sdd * Q1;                               // s_ddot q
  // step vector to the previous sample (x = rx - sin d, y = ry + cos d; cc.py:131-132)
  const double E0x = (i_rx - rowp[0]) - (i_sth * A0 - rowp[3] * rowp[8]), E1x = -(i_sth * B0 - rowp[3] * rowp[9]);
  const double E0y = (i_ry - rowp[1]) + (i_cth * A0 - rowp[2] * rowp[8]), E1y = i_cth * B0 - rowp[2] * rowp[9];
  const unsigned segmask = __match_any_sync(0xffffffffu, p);
  const bool seg_leader = (__ffs(segmask) - 1) == lane;
  const double kTan01Sq = 0.010067046422495888;                                // tan(0.1)^2
  unsigned* flags_p = flags + (active ? p : 0) * G.nw4;

  const double sd4 = sd2 * sd2;
  unsigned anyslow = 0u;
  // Three of the tests can be settled per ITEM for every lateral target at once, because the quantities are
  // affine / convex in d_i: the lateral offset d(d_i) is affine and fma is monotone, so max |d| sits at an end of
  // the grid (exact); the step vector is affine, so |step| <= |E0| + max|d_i| |E1| (teleport, checked with a
  // margin); v^2 = s_dot^2 (q^2 + d'^2) is convex, so its maximum is at an end (checked with a margin for the
  // rounding of the interior points).  When that holds for all items of a warp the loop below runs without
  // those tests; otherwise the warp runs the full chain.  Two more guards go the same way: q(d_i) = 1 - kappa_r d
  // is affine, so the singularity test q <= 0.05 is decided by the smaller end (exact), and when every coefficient
  // is finite and below 1e40 no intermediate of the chain can overflow, so the non-finite test cannot fire.
  // Together 13 of the 46 FP64-pipe instructions per candidate.
  bool lite, skip;
  {
    const double ga = brake_blk ? 0.0 : P.d_min, gb = brake_blk ? 0.0 : P.d_max, gabs = fmax(fabs(ga), fabs(gb));
    const double bx = fabs(E0x) + gabs * fabs(E1x), by = fabs(E0y) + gabs * fabs(E1y);
    const bool ok_tele = fma(bx, bx, by * by) <= 0.99 * tele2;
    const bool ok_road = fabs(fma(ga, B0, A0)) <= road_thr && fabs(fma(gb, B0, A0)) <= road_thr;
    const double qa = fma(ga, Q1, Q0), pa = fma(ga, P1, P0), qb = fma(gb, Q1, Q0), pb = fma(gb, P1, P0);
    const double vcap = vmax2 * (1.0 - 1e-12);
    const bool ok_speed = sd2 * fma(qa, qa, pa * pa) <= vcap && sd2 * fma(qb, qb, pb * pb) <= vcap;
    const bool ok_sing = fmin(qa, qb) > 0.05;
    const double mag = fabs(Q0) + fabs(P0) + fabs(R0) + fabs(M0) + fabs(S0) + sd2 + fabs(i_rk) +
                       gabs * (fabs(Q1) + fabs(P1) + fabs(R1) + fabs(M1) + fabs(S1));
    const bool ok_fin = mag <= 1e40;
    const bool lite_ok = ok_tele && ok_road && ok_speed && ok_sing && ok_fin;
    lite = __all_sync(0xffffffffu, !valid || lite_ok);                         // NaN anywhere: full chain
    // Interval screen of what is left (acceleration, curvature, lateral acceleration, the low-speed regime): with
    // q in [qmin, qmax] (positive here), |d'| <= Pm, |d''| <= Rm, ... every test is implied for ALL lateral targets
    // by one comparison of bounds.  Loose near the limits, but most items are far inside them: a warp whose items
    // all pass leaves every flag clear without looking at a single candidate.
    const double qmin = fmin(qa, qb), qmax = fmax(qa, qb), Pm = fmax(fabs(pa), fabs(pb));
    const double Rm = fmax(fabs(fma(ga, R1, R0)), fabs(fma(gb, R1, R0)));
    const double Mm = fmax(fabs(fma(ga, M1, M0)), fabs(fma(gb, M1, M0)));
    const double Sm = fmax(fabs(fma(ga, S1, S0)), fabs(fma(gb, S1, S0)));
    const double h2lo = qmin * qmin, h2hi = fma(qmax, qmax, Pm * Pm), ark = fabs(i_rk);
    const double Wm = fma(ark, h2hi, fma(Rm, qmax, Mm * Pm));                  // |kappa h^3|
    const double Tm = fma(Pm, fma(ark, h2hi, Wm), Mm * h2hi);
    const double Zm = fma(sd2, Tm, Sm * h2hi);                                 // |a h q|
    const double slack = 1.0 + 1e-9, Wm2 = Wm * Wm * slack;
    const bool ok_rest = Wm2 <= kmax2 * (h2lo * h2lo * h2lo) && sd4 * Wm2 <= latmax2 * h2lo &&
                         Zm * Zm * slack <= amax2 * (h2lo * h2lo) && sd2 * h2lo > 0.25 * slack;
    skip = __all_sync(0xffffffffu, !valid || (lite_ok && (!chk || ok_rest)));
#ifdef FOT_PHASE_CLOCKS
    {   // screen statistics: valid items, items that need the loop, warps with valid items (high word: full chain), skipped warps
      const unsigned bv = __ballot_sync(0xffffffffu, valid), bd_ = __ballot_sync(0xffffffffu, valid && !(lite_ok && (!chk || ok_rest)));
      const unsigned bl = __ballot_sync(0xffffffffu, valid && !lite_ok);
      if (lane == 0 && bv) {
        atomicAdd(&g_phase_clk[12], (unsigned long long)__popc(bv));
        atomicAdd(&g_phase_clk[13], (unsigned long long)__popc(bd_));
        atomicAdd(&g_phase_clk[14], 1ull | ((unsigned long long)(bl != 0) << 32));
        atomicAdd(&g_phase_clk[15], (unsigned long long)(bd_ == 0));
      }
    }
#endif
  }
  // one candidate sample, straight-line: flags of candidate i0 + U into byte U of acc
  auto sample = [&](auto lite_tag, double di, unsigned& acc, unsigned sh) {
    constexpr bool kLite = decltype(lite_tag)::value;
    const double qq = fma(di, Q1, Q0), dpr = fma(di, P1, P0), dpp = fma(di, R1, R0);
    const double m = fma(di, M1, M0), sq = fma(di, S1, S0);
    const double h2 = fma(qq, qq, dpr * dpr);                                  // hypot(q, d')^2 = (q / cos delta)^2
    const double w = fma(i_rk, h2, fma(dpp, qq, m * dpr));                     // kappa h^3   (cc.py:144-147)
    const double h6 = h2 * h2 * h2;
    const double w2 = w * w;
    const double v2 = sd2 * h2;                                                // v^2         (cc.py:150-152)
    const double T = fma(dpr, fma(-i_rk, h2, w), -(m * h2));
    const double Z = fma(sd2, T, sq * h2);                                     // a h q       (cc.py:155-157)
    const double acc_rhs = amax2 * (qq * qq * h2), curv_rhs = kmax2 * h6, lat_lhs = sd4 * w2, lat_rhs = latmax2 * h2;
    const double Z2 = Z * Z;
    if constexpr (kLite) {
      asm("{\n .reg .pred p, f;\n"
          " setp.gt.f64 f, %2, %3;\n"                                             // v > 0.5 (fp.py:1019)
          " @!f or.b32 %1, %1, 1;\n"
          " setp.gt.and.f64 p, %4, %5, f;\n"                                      // |kappa| > k_max when fast (fp.py:1020)
          " @p or.b32 %0, %0, %6;\n"
          "}"
          : "+r"(acc), "+r"(anyslow)
          : "d"(v2), "d"(fast2), "d"(w2), "d"(curv_rhs), "r"(F_CURV << sh));
    } else {
      const double ex = fma(di, E1x, E0x), ey = fma(di, E1y, E0y);
      const double step2 = fma(ex, ex, ey * ey);                               // fp.py:954 (squared)
      const double fin = fabs(Z) + fabs(w) + h6;
      asm("{\n .reg .pred p, f;\n .reg .f64 t;\n"
          " abs.f64 t, %2;\n setp.lt.f64 p, t, 0d7FF0000000000000;\n setp.le.and.f64 p, %2, 0d3FA999999999999A, p;\n"   // q <= 0.05 and finite (fp.py:826-833)
          " setp.geu.or.f64 p, %3, 0d7FF0000000000000, p;\n"                      // non-finite v / a / kappa (fp.py:944-946)
          " setp.gt.or.f64 p, %4, %5, p;\n"                                       // teleport (fp.py:953-956)
          " @p or.b32 %0, %0, %6;\n"
          " setp.gt.f64 f, %7, %8;\n"                                             // v > 0.5 (fp.py:1019)
          " @!f or.b32 %1, %1, 1;\n"
          " setp.gt.and.f64 p, %9, %10, f;\n"                                     // |kappa| > k_max when fast (fp.py:1020)
          " @p or.b32 %0, %0, %11;\n"
          "}"
          : "+r"(acc), "+r"(anyslow)
          : "d"(qq), "d"(fin), "d"(step2), "d"(tele2), "r"(F_DROP << sh), "d"(v2), "d"(fast2), "d"(w2), "d"(curv_rhs), "r"(F_CURV << sh));
      flag_gt(acc, v2, vmax2, F_SPEED << sh);                                  // fp.py:964
      flag_abs_gt(acc, fma(di, B0, A0), road_thr, F_ROAD << sh);               // fp.py:982
    }
    flag_gt(acc, Z2, acc_rhs, F_ACCEL << sh);                                  // fp.py:966
    flag_gt(acc, lat_lhs, lat_rhs, F_LAT << sh);                               // fp.py:975  v^2 |kappa| > a_lat
  };
  auto sweep_targets = [&](auto lite_tag) {
    for (int i0 = 0; i0 < n_dl; i0 += 4) {
      unsigned acc = 0u;
      if (valid) {
        if (brake_blk) {
          sample(lite_tag, 0.0, acc, 0u);
        } else if (i0 + 4 <= n_dl) {
          const double g0 = dgrid[i0], g1 = dgrid[i0 + 1], g2 = dgrid[i0 + 2], g3 = dgrid[i0 + 3];
          sample(lite_tag, g0, acc, 0u); sample(lite_tag, g1, acc, 8u); sample(lite_tag, g2, acc, 16u); sample(lite_tag, g3, acc, 24u);
        } else {
          for (int u = 0; i0 + u < n_dl; ++u) sample(lite_tag, dgrid[i0 + u], acc, 8u * u);
        }
      }
      const unsigned red = __reduce_or_sync(segmask, acc & keep4);
      if (seg_leader && active && red) atomicOr(&flags_p[i0 >> 2], red);
    }
  };
  if (skip) { }
  else if (lite) sweep_targets(std::true_type{});
  else sweep_targets(std::false_type{});
  // Low-speed regime (fp.py:1022-1032): items that saw a candidate with v <= 0.5 queue up; the block
  // redoes the two low-speed tests for them in phase D, one (item, candidate) unit per thread.
  if (anyslow && chk) slowq[atomicAdd(&s_nslow, 1)] = (unsigned short)tid;
  // Samples beyond the NaN prefix that are inside the spline domain again still count for the
  // candidate-wide singularity guard (fp.py:826-833 runs before the truncation).  Essentially never.
  if (active && !valid && i_rx == i_rx && keep > 0) {
    for (int i = 0; i < n_dl; ++i) {
      const double qq = fma(brake_blk ? 0.0 : dgrid[i], Q1, Q0);
      if ((qq <= 0.05) & (fabs(qq) < inf)) atomicOr(&flags_p[i >> 2], F_DROP << (8 * (i & 3)));
    }
  }
  // stop-distance directive (fp.py:307-324) needs v at the last kept sample
  if (stop_dist == stop_dist && valid && n == keep - 1) {
    for (int i = 0; i < n_dl; ++i) {
      const double di = brake_blk ? 0.0 : dgrid[i];
      const double qq = fma(di, Q1, Q0), dpr = fma(di, P1, P0);
      vlast[p * n_d + i] = sd2 * fma(qq, qq, dpr * dpr);
    }
  }
  asm volatile("cp.async.wait_all;" ::: "memory");   // cost-table entries of phase A have landed (visible after the barrier)
  FOT_PHASE_MARK(4);
  __syncthreads();
  FOT_PHASE_MARK(5);

  // ---- phase D: collision (fp.py:1035-1233) --------------------------------------------------------
  const int max_viol = dist_mode ? (int)floor(P.cfg.chance_epsilon * (double)B.S) : 0;   // fp.py:1114
  const bool budget = dist_mode && max_viol > 0;
  const int n_ls = s_nlist[0], n_ld = s_nlist[1];
  if (G.stage_dyn) mbar_wait(&s_bar, 0u);             // always: the copy must have landed before the block can exit
  {
    // low-speed tests of unit (queued item, candidate i): lateral step vs longitudinal step, heading
    // change vs the 0.1 rad / kappa_max * step floor (fp.py:1022-1032), from the item rows
    auto slow_unit = [&](int it, int i) {
      const int sp = it / N, sn = it - sp * N;
      // a candidate that already carries a flag of curvature priority or higher cannot change category
      if ((flags[sp * G.nw4 + (i >> 2)] >> (8 * (i & 3))) & (F_DROP | F_SPEED | F_ACCEL | F_CURV)) return;
      const double* r1 = row + (sp * NT + sn) * kRowW;                 // sample n
      const double* r0 = r1 - kRowW;                                           // sample n - 1 (only checked samples queue)
      const double di = brake_blk ? 0.0 : dgrid[i];
      const double d = fma(di, r1[9], r1[8]), dprev = fma(di, r0[9], r0[8]);
      const double qq = fma(-r1[4], d, 1.0), dpr = fma(di, r1[11], r1[10]) * r1[6];
      const double ssd = r1[7];
      if (ssd * ssd * fma(qq, qq, dpr * dpr) > 0.25) return;                   // this candidate is in the fast regime here
      bool badc;
      if (fabs(d - dprev) > fmax(1.5 * fabs(r1[5] - r0[5]), 0.02)) {
        badc = true;
      } else {
        // |wrap(yaw_n - yaw_{n-1})| is the angle between the heading vectors u = R(theta_r)(q, d')
        const double kmax = lim[2];
        const double q_prev = fma(-r0[4], dprev, 1.0);
        const double dp_prev = fma(di, r0[11], r0[10]) * r0[6];
        const double ux = r1[2] * qq - r1[3] * dpr, uy = r1[3] * qq + r1[2] * dpr;
        const double uxp = r0[2] * q_prev - r0[3] * dp_prev, uyp = r0[3] * q_prev + r0[2] * dp_prev;
        const double cr = uxp * uy - uyp * ux, dt_ = uxp * ux + uyp * uy;
        const double ex = fma(-r1[3], d, r1[0]) - fma(-r0[3], dprev, r0[0]);
        const double ey = fma(r1[2], d, r1[1]) - fma(r0[2], dprev, r0[1]);
        const double step2 = fma(ex, ex, ey * ey);
        if (kmax * kmax * step2 <= 0.01)
          // the threshold is the 0.1 rad floor: angle > 0.1 <=> dot <= 0 or cross^2 > tan(0.1)^2 dot^2
          badc = dt_ <= 0.0 || cr * cr > kTan01Sq * dt_ * dt_;
        else
          badc = fabs(atan2(cr, dt_)) > kmax * sqrt(step2);
      }
      if (badc) atomicOr(&flags[sp * G.nw4 + (i >> 2)], F_CURV << (8 * (i & 3)));
    };

    // clean masks: every thread needs its own pair's (cull decision + lateral window); the exact
    // tests read them from shared memory after the round's barrier
    unsigned cw_lo = 0u;
    int i_lo = -1, i_hi = -1;                            // lowest / highest clean candidate of the pair
    if (valid && n_ls + n_ld > 0)
      for (int w = 0; w < G.nwc; ++w) {
        const unsigned cwd = clean_word(flags_p, G.nw4, n_dl, w);
        if (cwd) { if (i_lo < 0) i_lo = 32 * w + __ffs(cwd) - 1; i_hi = 32 * w + 31 - __clz(cwd); }
        cw_lo |= cwd;
      }
    if (tid < n_k * G.nwc) {
      const int ap = tid / G.nwc, aw = tid - ap * G.nwc;
      const int afn = pi_fn[ap];
      cleanw[tid] = (afn == 0x7fffffff || afn >= 2) ? clean_word(flags + ap * G.nw4, G.nw4, n_dl, aw) : 0u;
    }
    const bool cull = valid && cw_lo != 0u;
    const int kob = B.T_obs > 0 ? min(n, B.T_obs - 1) : 0;                     // clip(round(t/dt)) = n (fp.py:1226-1227)
    // tangent-frame window: along = (o - ref).t within the collision radius, across = (o - ref).n within
    // the radius of the lateral offsets the pair's clean candidates take at this sample
    const double ca = fma(i_rx, i_cth, i_ry * i_sth), cn = fma(i_ry, i_cth, -(i_rx * i_sth));
    double d_lo = A0, d_hi = A0;
    if (cull && !brake_blk) {
      const double ga = P.d_sorted ? dgrid[i_lo] : P.d_min, gb = P.d_sorted ? dgrid[i_hi] : P.d_max;
      d_lo = A0 + fmin(ga * B0, gb * B0) - 1e-9;
      d_hi = A0 + fmax(ga * B0, gb * B0) + 1e-9;
    }
    int qsel = 0;

    // exact test of entry (item, obstacle) against every live clean candidate of the item's pair.
    // (Candidates the low-speed pass rejects in the same round may still be tested: harmless, the
    // curvature category outranks the collision category.)
    auto process = [&](int it, int e, bool queued) {
      const int ep = it / N, en = it - ep * N;
      const bool is_dyn = e >= n_ls;
      const unsigned off = is_dyn ? olist[M + e - n_ls] : olist[e];
      const unsigned ok_ = off + (unsigned)(B.T_obs > 0 ? min(en, B.T_obs - 1) : 0);
      const double2 o = is_dyn ? (G.stage_dyn ? dynst[ok_] : dyn_q[ok_]) : stat_q[off];
      const double r2 = is_dyn ? r2_dyn : P.cfg.collide_r2;
      const bool use_budget = budget && is_dyn;
      const double* r = row + (ep * NT + en) * kRowW;
      const double cth = r[2], sth = r[3];
      const double X0 = fma(-sth, r[8], r[0]) - o.x, X1 = -(sth * r[9]);       // x - ox = X0 + d_i X1
      const double Y0 = fma(cth, r[8], r[1]) - o.y, Y1 = cth * r[9];
      for (int w = 0; w < G.nwc; ++w) {
        // from the queue: the masks were published before the round's barrier; in place (queue full, before that
        // barrier): this thread's own pair, recomputed from the flags, which are final since the previous barrier
        unsigned mbits = queued ? cleanw[ep * G.nwc + w] : clean_word(flags + ep * G.nw4, G.nw4, n_dl, w);
        if (!use_budget) mbits &= ~hitw[ep * G.nwc + w];
        while (mbits) {
          const int bit = __ffs(mbits) - 1;
          mbits &= mbits - 1u;
          const int i = w * 32 + bit;
          const double di = brake_blk ? 0.0 : dgrid[i];
          bool hit = false;
          if (n_circ == 0) {
            const double dx = fma(di, X1, X0), dy = fma(di, Y1, Y0);
            hit = dx * dx + dy * dy <= r2;                                     // fp.py:1196-1198, :1231-1233
          } else {                                                             // fp.py:1158-1167
            const double d = fma(di, r[9], r[8]);
            const double dpr = fma(di, r[11], r[10]) * r[6];
            const double qq = fma(-r[4], d, 1.0);
            const double rh = 1.0 / sqrt(fma(qq, qq, dpr * dpr));
            const double hx = (cth * qq - sth * dpr) * rh, hy = (sth * qq + cth * dpr) * rh;   // (cos yaw, sin yaw)
            for (int ci = 0; ci < n_circ && !hit; ++ci) {
              const double dx = fma(di, X1, X0) + P.cfg.circle_offsets[ci] * hx, dy = fma(di, Y1, Y0) + P.cfg.circle_offsets[ci] * hy;
              hit = dx * dx + dy * dy <= r2;
            }
          }
          if (hit) {
            if (!use_budget) atomicOr(&hitw[ep * G.nwc + w], 1u << bit);
            else { const int sidx = (int)(off / (unsigned)B.T_obs) / B.P; atomicOr(&viol[(ep * n_d + i) * G.vwords + (sidx >> 5)], 1u << (sidx & 31)); }
          }
        }
      }
    };

    // window test of this item against list entries [ea, eb) of one kind; survivors -> queue
    auto cull_range = [&](auto dyn_tag, auto stage_tag, int ea, int eb, int e0) {
      constexpr bool kDyn = decltype(dyn_tag)::value;
      constexpr bool kStaged = decltype(stage_tag)::value;
      const double2* obs_k = (kStaged ? dynst : dyn_q) + kob;                  // this item's time step
      const double rc = kDyn ? rc_d : rc_s;
      const double w_lo = d_lo - rc, w_hi = d_hi + rc;
      const unsigned* lst = kDyn ? olist + M - n_ls : olist;                   // entry e -> lst[e]
      for (int e32 = ea; e32 < eb; e32 += 32) {
        const int ee = min(eb, e32 + 32);
        unsigned rel = 0u, bit = 1u;
#pragma unroll 4
        for (int e = e32; e < ee; ++e, bit <<= 1) {
          const double2 o = kDyn ? obs_k[lst[e]] : stat_q[lst[e]];
          const double al = fma(o.x, i_cth, fma(o.y, i_sth, -ca));
          const double ac = fma(o.y, i_cth, fma(-o.x, i_sth, -cn));
          if ((fabs(al) <= rc) & (ac >= w_lo) & (ac <= w_hi)) rel |= bit;      // NaN -> false
        }
        while (rel) {
          const int e = e32 + __ffs(rel) - 1;
          rel &= rel - 1u;
          const int slot = atomicAdd(&s_qcount[qsel], 1);
          if (slot < G.qcap) queue[slot] = ((unsigned)tid << 16) | (unsigned)(e - e0);
          else process(tid, e, false);                                         // queue full: test right here
        }
      }
    };

    const int n_l = n_ls + n_ld;
    int e0 = 0;
    do {                                                 // at least one round: it also drains the low-speed queue
      const int e1 = min(n_l, e0 + G.ochunk);
      if (cull) {
        if (e0 < n_ls) cull_range(std::false_type{}, std::false_type{}, e0, min(e1, n_ls), e0);
        if (e1 > n_ls) {
          if (G.stage_dyn) cull_range(std::true_type{}, std::true_type{}, max(e0, n_ls), e1, e0);
          else cull_range(std::true_type{}, std::false_type{}, max(e0, n_ls), e1, e0);
        }
      }
      FOT_PHASE_MARK(6);
      __syncthreads();
      FOT_PHASE_MARK(7);
      const int cnt = min(s_qcount[qsel], G.qcap);
      if (tid == 0) s_qcount[qsel ^ 1] = 0;
      // queue entries first (their cost varies with the number of live candidates), then the low-speed
      // units; warps fetch 32 units at a time from a shared counter so that a warp stuck with long entries
      // does not hold the block back
      const int n_units = cnt + (e0 == 0 ? s_nslow * n_dl : 0);
      for (;;) {
        int base = 0;
        if (lane == 0) base = atomicAdd(&s_next[qsel], 32);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= n_units) break;
        const int u = base + lane;
        if (u < cnt) {
          const unsigned ent = queue[u];
          process((int)(ent >> 16), e0 + (int)(ent & 0xffffu), true);
        } else if (u < n_units) {
          const int k = (u - cnt) / n_dl;
          slow_unit(slowq[k], (u - cnt) - k * n_dl);
        }
      }
      if (tid == 0) s_next[qsel ^ 1] = 0;
      qsel ^= 1;
      e0 = e1;
      if (e1 < n_l && !budget) {
        // leave early once every clean candidate of the block has its decisive hit
        bool alive = false;
        if (tid < n_k * G.nwc) {
          alive = (cleanw[tid] & ~hitw[tid]) != 0u;
        }
        if (!__syncthreads_or(alive ? 1 : 0)) break;
      } else {
        FOT_PHASE_MARK(8);
        __syncthreads();
        FOT_PHASE_MARK(9);
      }
    } while (e0 < n_l);
  }

  // ---- phase E: category, cost, block arg-min, histogram ----------------------------------------
  for (int c = tid; c < n_cand; c += bd) {
    const int cp = c / n_dl, ci = c - cp * n_dl;
    const int li = brake_blk ? cp : ci;
    // cost on the un-truncated profile (fp.py:703-734)
    // jerk sums and terminal offsets from fot_prepass (staged in phase A)
    const double Js = ctb[cp], Jp = ctb[G.pcap + li], d_end = ctb[G.pcap + G.ct_lcap + li];
    const double Jd = d_end * d_end;
    const double dv = B.target[q] - sdl[cp];
    const double Jv = dv * dv;
    const double Jt = (double)(N - 1) * dt;
    const double lat_cost = P.cfg.k_j * Jp + P.cfg.k_t * Jt + P.cfg.k_d * Jd;
    const double lon_cost = P.cfg.k_j * Js + P.cfg.k_t * Jt + P.cfg.k_s_dot * Jv;
    const double cost = P.cfg.k_lat * lat_cost + P.cfg.k_lon * lon_cost;
    const unsigned byte = (flags[cp * G.nw4 + (ci >> 2)] >> (8 * (ci & 3))) & 0xffu;
    const int cfn = pi_fn[cp];
    const int ckeep = cfn == 0x7fffffff ? N : (cfn >= 2 ? cfn : 0);
    int cat;
    if (ckeep == 0 || (byte & F_DROP)) cat = FOT_CAT_DROP;                     // fp.py:831-833, :933, :944, :953
    else if (byte & F_SPEED) cat = FOT_CAT_SPEED;
    else if (byte & F_ACCEL) cat = FOT_CAT_ACCEL;
    else if (byte & F_CURV) cat = FOT_CAT_CURV;
    else if (byte & F_LAT) cat = FOT_CAT_LAT;
    else if (byte & F_ROAD) cat = FOT_CAT_ROAD;
    else {
      bool hit = (hitw[cp * G.nwc + (ci >> 5)] >> (ci & 31)) & 1u;
      if (G.vwords > 0) {
        int nv = 0;
        for (int w = 0; w < G.vwords; ++w) nv += __popc(viol[(cp * n_d + ci) * G.vwords + w]);
        hit = hit || nv > max_viol;                                            // fp.py:1113-1124
      }
      if (hit) {
        cat = FOT_CAT_COLL;                                                    // fp.py:986-989
      } else {
        cat = FOT_CAT_OK;
        if (stop_dist == stop_dist) {                                          // fp.py:307-324
          const double v_last = sqrt(vlast[cp * n_d + ci]);
          const double s_span = row[(cp * NT + ckeep - 1) * kRowW + 5] - row[cp * NT * kRowW + 5];
          if (!(v_last <= 0.15 && s_span <= stop_dist + 1e-6)) cat = FOT_CAT_STOP;
        }
      }
    }
    const int cand_idx = cand0 + c;
    if (cat < FOT_N_STATS) atomicAdd(&s_stats[cat], 1);
    if (O.cand_cat) O.cand_cat[(size_t)q * O.cand_stride + cand_idx] = (uint8_t)cat;
    if (O.cand_cost) O.cand_cost[(size_t)q * O.cand_stride + cand_idx] = cost;
    if (cat == FOT_CAT_OK && cost < INFINITY) argmin_merge(my_cost, my_idx, cost, cand_idx);
  }
  FOT_PHASE_MARK(10);
  __syncthreads();                                       // this block's tables are dead; the next block may overwrite them
  FOT_PHASE_MARK(11);
  }  // blocks of this CTA

  if (G.stage_dyn && state_ok) mbar_wait(&s_bar, 0u);    // the bulk copy must have landed before the CTA can exit
  for (int off = 16; off > 0; off >>= 1) {
    const double oc = __shfl_down_sync(0xffffffffu, my_cost, off);
    const int oi = __shfl_down_sync(0xffffffffu, my_idx, off);
    argmin_merge(my_cost, my_idx, oc, oi);
  }
  if (lane == 0) { s_cost[tid >> 5] = my_cost; s_idx[tid >> 5] = my_idx; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < (bd >> 5); ++w) argmin_merge(my_cost, my_idx, s_cost[w], s_idx[w]);
    O.part_cost[part] = my_cost;
    O.part_idx[part] = (my_idx == 0x7fffffff) ? -1 : my_idx;
  }
  if (tid < FOT_N_STATS && s_stats[tid] != 0) atomicAdd(&O.stats[(size_t)q * FOT_N_STATS + tid], s_stats[tid]);
}

}  // namespace fot
