// fot_sweep_pairs.cuh -- the pair-per-warp sweep kernel (sm_100a, fp64).
//
// Same contract and the same arithmetic as fot_sweep_items (fot_sweep_items.cuh): every candidate's validity
// flags, collision verdict, category and cost come out bit-identical.  What changes is who waits for whom.
// fot_sweep_items cuts a query into blocks of six longitudinal profiles and walks its 320 threads through six
// block-wide barriers per block; ncu charges 3.1 stall cycles per issued instruction to those barriers, and
// a two-barrier variant (fewer barriers, a shared producer/consumer queue; DESIGN.md section 4c) only moved the wait
// into the queue.  Here the
// unit of work is ONE PAIR = one longitudinal profile (horizon T_j, terminal speed v_k) or one brake horizon,
// and a pair belongs to ONE WARP from its first instruction to its last:
//
//   CTA    = one query (or 1/ctas_per_query of its pairs for small batches): obstacle block staged once by a
//            bulk copy, spline tables, lateral grid and the query's scalars in shared memory;
//   warp   = fetches the next pair of the query from a shared counter (longest horizons first) and does everything
//            for it -- item set-up, validity chain, low-speed tests, obstacle list, window cull, exact distance
//            tests, category, cost, arg-min -- out of a private slice of shared memory;
//   lane   = sample t_n of the pair (passes of 32 samples); the loop runs over the lateral targets d_i.
//
// There is no __syncthreads() between the CTA's set-up and its final arg-min: warps never wait for each other,
// the phases of different warps decorrelate (one warp's latency-bound set-up chain overlaps another's FP64-bound
// validity loop), and an expensive pair delays nobody.  Because all 32 lanes of a warp work on the same pair,
// the per-candidate state is warp-uniform: flags are OR-reduced by one `redux` and stored by one lane without
// atomics, the clean masks and decisive-hit words are plain words, the survivor queue is filled by ballot +
// prefix count, and the exact tests run a uniform loop over the live candidates with one ballot each.
//
// What that bought and what it cost is in DESIGN.md section 4d: the barrier stall went from 3.1 to 0.4 cycles per issued
// instruction, and the first version was slower for it -- twenty warps that each walk their own way through 30-40 KB of
// mostly straight-line code do not share instruction fetches the way ten warps in lock-step do.  From then on the kernel's
// time followed the size of its hot code (profiles/r2/sweep_pairs_icache_history.txt), which is why the slice layout is a
// compile-time constant, why there is one code site per job in the collision loop, and why the batch shape of a planning
// campaign has an instantiation of its own (kFeat = 0) with every other mode compiled out.
//
// The upload gate, the boxes of a staged obstacle block, the reference point and the flag idiom are the functions of
// fot_sweep_math.cuh that fot_sweep_items calls too.  Reference citations as in fot_sweep_items.cuh (fp.py = src/planning/frenet_planner.py, cs.py = cubic_spline.py,
// cc.py = src/core/coordinate_converter.py).
#pragma once
#include <cstddef>
#include <type_traits>
#include "fot_sweep_math.cuh"

namespace fot {

#ifndef FOT_PAIR_THREADS
#define FOT_PAIR_THREADS 320
#endif
#ifndef FOT_PAIR_MIN_CTAS
#define FOT_PAIR_MIN_CTAS 2
#endif
constexpr int kPairThreads = FOT_PAIR_THREADS;   // CTA size of fot_sweep_pairs
constexpr int kPairWarps = kPairThreads / 32;
constexpr int kPairList = 64;                    // obstacle list entries per chunk (per warp): dynamic from the front, static from the back
constexpr int kPairQueue = 64;                   // survivor queue (per warp, a ring): < 32 waiting + <= 32 new
#ifndef FOT_PAIR_NT
#define FOT_PAIR_NT 56
#endif
constexpr int kPairNT = FOT_PAIR_NT;             // samples per profile this kernel covers (longer time grids: fot_sweep_items)
constexpr int kPairND = 96;                      // lateral targets this kernel covers (wider grids: fot_sweep_items)
constexpr int kPairNV = 52;                      // terminal speeds per query
constexpr int kPairNX = 48;                      // spline knots (longer reference lines: fot_sweep_items)
constexpr int kPairNH = 64;                      // horizons

// One warp's private slice of shared memory, and behind the slices the CTA-wide tables whose size has a small bound.
// The layout is a compile-time constant on purpose: every access is `base register + immediate`.  (With run-time
// offsets the compiler rebuilt the addresses from the thread index at every use -- a fifth of the hot instructions of
// the first version of this kernel, which is bound by instruction fetch.)
struct __align__(16) PairSlice {
  double row[kRowW][kPairNT];          // item rows of the current pair, field-major: rx ry cos sin | kappa s 1/s_dot s_dot | A0 B0 A1 B1
                                       // (lane = sample reads and writes are conflict-free)
  unsigned flags[kPairND / 4];         // validity flags, one byte per candidate
  unsigned hitw[4];                    // decisive collision, one bit per candidate
  unsigned cleanw[4];                  // kinematically clean
  unsigned wl[kPairList];              // obstacle list: element offsets; dynamic entries from the front (padded to a multiple
                                       // of four), static entries (bit 31 set) from the back
  unsigned q_off[kPairQueue];          // survivor queue: obstacle element offset
  unsigned char q_n[kPairQueue];       //                 sample
  unsigned short slowq[kPairNT];       // samples with a low-speed candidate
  double pc[16];                       // the pair's polynomials: quartic a0..a4 | lateral basis c0..c5, b3..b5 | hold
};
struct __align__(16) PairShared {
  PairSlice w[kPairWarps];
  double qc[12 + kPairNV];             // fs[6] | limits[4] | target | stop_dist | v_grid[n_v]
  double dgrid[kPairND + 2];           // lateral targets, then the brake ladder's single target 0.0
  double spl[9][kPairNX];              // spline tables: knots | x: a b c d | y: a b c d
  int n_steps[kPairNH];                // samples - 1 of every horizon
};

static_assert(offsetof(PairSlice, hitw) == offsetof(PairSlice, flags) + kPairND && offsetof(PairSlice, cleanw) == offsetof(PairSlice, hitw) + 16 &&
              kPairND / 4 + 8 == 32, "flags | hitw | cleanw are zeroed as 32 consecutive words");

struct PairGeom {
  int32_t ctas_per_query;    // CTAs that share one query's pairs (1 in large batches)
  int32_t nw4, nwc, vwords;  // flag words (4 candidates each) / mask words (32 candidates each) / violation words per candidate
  int32_t stage_dyn;         // 1: the query's obstacle block is staged in shared memory by one bulk copy
  int32_t box_smem;          // 1: trajectory boxes in shared memory (copied from fot_prepass, or built here when fused_box)
  int32_t fused_box;         // 1: boxes built by the CTA from its staged block (gated host-pointer call)
  // byte offsets into dynamic shared memory of the run-time sized tables (behind PairShared)
  int32_t o_dyn, o_box, o_viol;
  int32_t viol_bytes;        // per warp: [n_d][vwords] violation bitmaps (chance-constrained mode with a budget)
  // gated launch (see ItemGeom)
  int32_t gate_q0, gate_per;
  uint32_t gate_epoch;
  unsigned* gate;
};

// spline_ref_tab over the shared-memory tables of PairShared: compile-time strides.
struct SmemSplineTab {
  const double (*T)[kPairNX];
  __device__ __forceinline__ double operator()(int k, int i) const { return T[k][i]; }
};
// kFused: the variant of the gated host-pointer call (waits for its query's upload slice, boxes the trajectories itself).
// kFeat: which optional modes this instantiation carries (PAIR_*).  The kernel is bound by instruction fetch (DESIGN.md
// section 4d), so the code of a mode the batch does not use is compiled out of the instantiation it runs instead of
// being branched over: 0 is the shape of a planning campaign (no static obstacles, one collision circle, no violation
// budget, sorted lateral grid, staged obstacle block, no per-candidate outputs); the host picks the smallest
// instantiated superset of what the batch needs (fot_api.cu, kPairInstances).  PAIR_ROUTES: every query on its own
// reference path (Batch::rt, DESIGN.md section 4h) -- the CTA copies that route's tables and keeps its knot count in a
// register; PAIR_ALL is every mode but this one.
enum : int { PAIR_STATIC = 1, PAIR_FOOTPRINT = 2, PAIR_BUDGET = 4, PAIR_OUTPUTS = 8, PAIR_LOOSE = 16, PAIR_ALL = 31,
             PAIR_ROUTES = 32 };
template <bool kFused, int kFeat>
__global__ void __launch_bounds__(kPairThreads, FOT_PAIR_MIN_CTAS)
fot_sweep_pairs(const Plan P, const Batch B, const Out O_, const PairGeom G) {
  Out O = O_;
  if (!(kFeat & PAIR_OUTPUTS)) { O.cand_cat = nullptr; O.cand_cost = nullptr; }
  extern __shared__ __align__(16) unsigned char smb[];
  PairShared& S = *reinterpret_cast<PairShared*>(smb);
  double* qc = S.qc;
  double* dgrid = S.dgrid;
  const double2* dynst = reinterpret_cast<const double2*>(smb + G.o_dyn);   // [SP][T_obs] when stage_dyn
  float4* sbox = reinterpret_cast<float4*>(smb + G.o_box);     // [SP] trajectory boxes when box_smem
  __shared__ int s_next;                 // next pair of this CTA
  __shared__ int s_stats[FOT_N_STATS];
  __shared__ double s_cost[kPairWarps];
  __shared__ int s_idx[kPairWarps];
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ int s_abort;

  const int NT = P.n_t_max;
  const int q = blockIdx.x / G.ctas_per_query;
  const int cta = blockIdx.x - q * G.ctas_per_query;
  const int tid = threadIdx.x, bd = blockDim.x;
  int lane = tid & 31, wid = tid >> 5;
  // opaque to the optimiser: held in registers instead of being rebuilt from %tid at every use
  unsigned wofs = (unsigned)wid * (unsigned)sizeof(PairSlice);
  asm volatile("" : "+r"(lane), "+r"(wofs));
  const unsigned full = 0xffffffffu, lt_mask = (1u << lane) - 1u;
  const double* fsg = B.frenet + 6 * (size_t)q;
  const int n_v = B.n_v[q];
  const int n_d = P.cfg.n_d;
  const double dt = P.cfg.dt;
  const size_t part = (size_t)q * G.ctas_per_query + cta;

  const bool has_dyn = B.dyn_raw != nullptr;
  const int SP = has_dyn ? B.S * B.P : 0;
  const int M = (kFeat & PAIR_STATIC) ? (B.static_raw ? B.n_static : 0) : 0;
  const double2* dyn_q = has_dyn ? reinterpret_cast<const double2*>(B.dyn_raw) + (size_t)q * SP * B.T_obs : nullptr;
  const double2* stat_q = M > 0 ? reinterpret_cast<const double2*>(B.static_raw) + (size_t)(B.static_per_query ? q : 0) * M : nullptr;

  // this warp's private slice
  PairSlice& W = *reinterpret_cast<PairSlice*>(smb + wofs);
  auto R = [&](int f, int n_) -> double& { return W.row[f][n_]; };
  unsigned* flags = W.flags;
  unsigned* hitw = W.hitw;
  unsigned* cleanw = W.cleanw;
  unsigned* wl = W.wl;
  unsigned* q_off = W.q_off;
  unsigned char* q_n = W.q_n;
  unsigned short* slowq = W.slowq;
  unsigned* viol = reinterpret_cast<unsigned*>(smb + G.o_viol + wid * G.viol_bytes);   // [n_d][vwords] (budget mode)
  (void)NT;

  // ---- once per CTA ---------------------------------------------------------------------------------
  Plan PR_;                                                 // PAIR_ROUTES: the query's route (route_plan, below)
  const Plan& PS = (kFeat & PAIR_ROUTES) ? PR_ : P;        // spline tables and knot count of this query
  if (kFused && G.gate && gate_wait(G, q, s_abort)) return;
  // PAIR_LOOSE: obstacle block read from global memory, boxes from global memory, or an unsorted lateral grid
  const bool stage_dyn = !(kFeat & PAIR_LOOSE) || G.stage_dyn, box_smem = !(kFeat & PAIR_LOOSE) || G.box_smem, d_sorted = !(kFeat & PAIR_LOOSE) || P.d_sorted;
  const int vwords = (kFeat & PAIR_BUDGET) ? G.vwords : 0;
  // Nothing below depends on a global load before the barrier: the CTA's first round trip to memory (Frenet state,
  // limits, speed grid, lateral grid, spline tables, trajectory boxes) is ONE, issued by all threads at once, and the bulk
  // copy of the obstacle block is in flight beside it.
  const bool staged = stage_dyn && SP > 0;
  if (tid == 0) {
    if (staged) {
      mbar_init(&s_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      const uint32_t bytes = (uint32_t)SP * (uint32_t)B.T_obs * 16u;
      mbar_expect_tx(&s_bar, bytes);
      tma_bulk_g2s(smb + G.o_dyn, dyn_q, bytes, &s_bar);
    }
    s_next = 0;
  }
  if (tid < FOT_N_STATS) s_stats[tid] = 0;
  for (int i = tid; i < P.cfg.n_T; i += bd) S.n_steps[i] = P.n_steps[i];
  for (int i = tid; i <= n_d; i += bd) dgrid[i] = i < n_d ? P.d_grid[i] : 0.0;   // [n_d]: the brake ladder's single target
  if (tid < 6) qc[tid] = fsg[tid];
  else if (tid < 10) qc[tid] = B.limits[4 * (size_t)q + tid - 6];
  else if (tid == 10) qc[10] = B.target[q];
  else if (tid == 11) qc[11] = B.stop_dist[q];
  for (int i = tid; i < B.n_v_max; i += bd) qc[12 + i] = B.v_grid[(size_t)q * B.n_v_max + i];
  if constexpr ((kFeat & PAIR_ROUTES) != 0) {
    // the route's id is read beside the other per-query loads, behind the bulk copy; a bad id plans nothing (the
    // copy must have landed before the CTA exits; thread 0 initialised the barrier and waits on it)
    if (!route_plan(P, B.rt, q, PR_)) {
      if (tid == 0) {
        if (staged) mbar_wait(&s_bar, 0u);
        O.part_cost[part] = INFINITY; O.part_idx[part] = -1;
      }
      return;
    }
  }
  {
    const int nx = PS.cfg.nx;
    for (int i = tid; i < nx; i += bd) {
      S.spl[0][i] = PS.knots[i];
      S.spl[1][i] = PS.xa[i];  S.spl[3][i] = PS.xc[i];
      S.spl[5][i] = PS.ya[i];  S.spl[7][i] = PS.yc[i];
      if (i < nx - 1) {
        S.spl[2][i] = PS.xb[i]; S.spl[4][i] = PS.xd[i];
        S.spl[6][i] = PS.yb[i]; S.spl[8][i] = PS.yd[i];
      }
    }
  }
  if (box_smem && !G.fused_box)
    for (int j = tid; j < SP; j += bd) sbox[j] = B.dyn_box[(size_t)q * SP + j];
  __syncthreads();
  // A non-finite Frenet state makes every sample of every candidate non-finite: the reference drops
  // them all silently (empty / non-finite guards fp.py:933-946).
  const bool state_ok = fabs(qc[0]) + fabs(qc[1]) + fabs(qc[2]) + fabs(qc[3]) + fabs(qc[4]) + fabs(qc[5]) < INFINITY;
  if (kFused && G.fused_box && staged) {
    // box every predicted trajectory of the staged obstacle block
    mbar_wait(&s_bar, 0u);
    box_staged(dynst, sbox, SP, B.T_obs, wid, bd >> 5, lane);
    __syncthreads();
  }

  const double* fs = qc;                 // the query's Frenet state, from shared memory
  const double* lim = qc + 6;
  const bool brake_on = fs[1] > 0.1 && P.cfg.n_B > 0;                          // fp.py:469 BRAKE_MIN_SPEED
  const int n_grid = P.cfg.n_T * n_v;
  const int n_units = n_grid + (brake_on ? P.cfg.n_B : 0);
  const float rcp_nv = 1.0f / (float)n_v;

  if (!state_ok) {
    if (O.cand_cat || O.cand_cost) {
      const int n_all = n_grid * n_d + (brake_on ? P.cfg.n_B : 0);
      for (int c = cta * bd + tid; c < n_all; c += G.ctas_per_query * bd) {
        if (O.cand_cat) O.cand_cat[(size_t)q * O.cand_stride + c] = (uint8_t)FOT_CAT_DROP;
        if (O.cand_cost) O.cand_cost[(size_t)q * O.cand_stride + c] = qnan();
      }
    }
    if (tid == 0) { O.part_cost[part] = INFINITY; O.part_idx[part] = -1; }
    if (staged) mbar_wait(&s_bar, 0u);                     // the bulk copy must have landed before the CTA can exit
    return;
  }

  // ---- per-CTA constants of the validity chain and the collision tests -----------------------------
  const int n_circ = (kFeat & PAIR_FOOTPRINT) ? P.cfg.n_circles : 0;
  double max_off = 0.0;                                  // footprint circles sit within max|offset| of the path point
  for (int i = 0; i < n_circ; ++i) max_off = fmax(max_off, fabs(P.cfg.circle_offsets[i]));
  const bool dist_mode = (B.dyn_mode == FOT_DYN_DISTRIBUTION);
  const double r2_dyn = dist_mode ? P.cfg.collide_r2 : P.cfg.collide_r2_single;   // fp.py:1099-1104, :1173
  const double rc_s = sqrt(P.cfg.collide_r2) * (1.0 + 1e-9) + 1e-9 + max_off;
  const double rc_d = sqrt(r2_dyn) * (1.0 + 1e-9) + 1e-9 + max_off;
  const double wroad = fmax(P.cfg.max_road_width + 1e-9, fabs(fs[3]));
  const float pad = __double2float_ru(wroad + fmax(rc_s, rc_d));
  const int max_viol = dist_mode ? (int)floor(P.cfg.chance_epsilon * (double)B.S) : 0;   // fp.py:1114
  const bool budget = (kFeat & PAIR_BUDGET) && dist_mode && max_viol > 0;
  const double inf = INFINITY;
  // squared limits; a negative limit rejects every checked sample, as `x > negative` does in the reference
  // (warp-uniform: pushed through redux so that they live in uniform registers)
  auto uni = [&](double x) {
    const unsigned lo = __reduce_or_sync(full, (unsigned)__double2loint(x));
    const unsigned hi = __reduce_or_sync(full, (unsigned)__double2hiint(x));
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
  const double stop_dist = qc[11];
  const double kTan01Sq = 0.010067046422495888;                                // tan(0.1)^2
  const float4* boxes = box_smem ? sbox : B.dyn_box + (size_t)q * SP;

  double my_cost = INFINITY;             // running arg-min over every pair this lane has seen
  int my_idx = 0x7fffffff;
  bool dyn_ready = !staged || (kFused && G.fused_box);

  for (;;) {
    // ---- next pair of this CTA: longest horizons first, the brake ladder last ----------------------
    int fetch = 0;
    if (lane == 0) fetch = atomicAdd(&s_next, 1);
    fetch = __shfl_sync(full, fetch, 0);
    const int ord = cta + fetch * G.ctas_per_query;
    if (ord >= n_units) break;
    const bool brake = ord >= n_grid;
    int jT = 0, kk, N, n_dl;
    if (!brake) {
      const int u = n_grid - 1 - ord;
      jT = __float2int_rz(((float)u + 0.5f) * rcp_nv);      // u / n_v (exact: u < 2^20)
      kk = u - jT * n_v;
      N = S.n_steps[jT] + 1;
      n_dl = n_d;
    } else {
      kk = ord - n_grid;
      N = P.cfg.n_total;
      n_dl = 1;
    }
    const int cand0 = brake ? n_grid * n_d + kk : (jT * n_v + kk) * n_d;      // generation order (fp.py:398-449)
    const double* dg = dgrid + (brake ? n_d : 0);             // lateral targets of this pair (brake: the single 0.0 slot)

    // ---- phase A: the pair's private state, its polynomials --------------------------------------------
    flags[lane] = 0u;                                       // flags | hit words | clean words (32 words in a row)
    if (vwords > 0)
      for (int i = lane; i < n_d * vwords; i += 32) viol[i] = 0u;
    {
      // quartic solve of the pair (fp.py:619-647) and the lateral basis: d_i(t) = A(t) + d_i * B(t) -- the quintic's
      // right-hand side is linear in the target (fp.py:676-683).  Once per pair; the passes reload the sixteen numbers.
      Lon L;
      double c0, c1, c2, c3, c4, c5, b3, b4, b5;
      if (!brake) {
        const double T = P.T[jT];
        L = lon_solve(fs, qc[12 + kk], T, P.inv4 + 4 * jT, n_v == 1, N - 1);
        const double* Ai = P.inv5 + 9 * jT;
        c0 = fs[3]; c1 = fs[4]; c2 = fs[5] / 2.0;
        const double r0 = -c0 - c1 * T - c2 * T * T, r1 = -c1 - 2.0 * c2 * T, r2 = -2.0 * c2;
        c3 = fma(r2, Ai[2], fma(r1, Ai[1], r0 * Ai[0]));
        c4 = fma(r2, Ai[5], fma(r1, Ai[4], r0 * Ai[3]));
        c5 = fma(r2, Ai[8], fma(r1, Ai[7], r0 * Ai[6]));
        b3 = Ai[0]; b4 = Ai[3]; b5 = Ai[6];
      } else {                                                                     // one lateral profile per brake horizon (fp.py:480-482)
        L = lon_solve(fs, 0.0, P.Tb[kk], P.inv4b + 4 * kk, true, P.n_steps_b[kk]);
        const Lat Lb = lat_solve(fs, fs[3], P.Tb[kk], P.inv5b + 9 * kk, true, P.n_steps_b[kk]);
        c0 = Lb.a0; c1 = Lb.a1; c2 = Lb.a2; c3 = Lb.a3; c4 = Lb.a4; c5 = Lb.a5;
        b3 = b4 = b5 = 0.0;
      }
      if (lane == 0) {
        double* pc = W.pc;
        pc[0] = L.a0; pc[1] = L.a1; pc[2] = L.a2; pc[3] = L.a3; pc[4] = L.a4;
        pc[5] = c0; pc[6] = c1; pc[7] = c2; pc[8] = c3; pc[9] = c4; pc[10] = c5; pc[11] = b3; pc[12] = b4; pc[13] = b5;
        pc[14] = __longlong_as_double((long long)L.hold);
      }
    }
    __syncwarp();

    // ---- phases B + C, 32 samples at a time ---------------------------------------------------------
    int fn = 0x7fffffff;                                   // first sample with a NaN reference point
    int nslow = 0;
    unsigned bxlo = 0xffffffffu, bxhi = 0u, bylo = 0xffffffffu, byhi = 0u;    // box of the reference points (ordered-uint floats)
    for (int n0 = 0; n0 < N; n0 += 32) {
      const int n = min(n0 + lane, N - 1);                   // lanes beyond the last sample repeat it (nothing of theirs is used)
      const bool active = n0 + lane < N;
      double i_rx, i_ry, i_cth, i_sth, i_rk, i_rdk, i_sd, i_sdd, i_isd;
      double A0, B0, A1, B1, A2, B2;
      {
        const double* pc = W.pc;
        const int hold = (int)__double_as_longlong(pc[14]);
        const bool held = n > hold;                                                // fp.py:487-499 brake padding
        const TPow tp = tpow(held ? hold : n, dt);
        const double s = pc[0] + pc[1] * tp.t + pc[2] * tp.t2 + pc[3] * tp.t3 + pc[4] * tp.t4;             // fp.py:644
        i_sd = held ? 0.0 : pc[1] + 2.0 * pc[2] * tp.t + 3.0 * pc[3] * tp.t2 + 4.0 * pc[4] * tp.t3;       // fp.py:645
        i_sdd = held ? 0.0 : 2.0 * pc[2] + 6.0 * pc[3] * tp.t + 12.0 * pc[4] * tp.t2;                      // fp.py:646
        const RefFast rp = spline_ref_tab(SmemSplineTab{S.spl}, PS.cfg.nx, s);
        i_rx = rp.rx; i_ry = rp.ry; i_cth = rp.cth; i_sth = rp.sth; i_rk = rp.rk; i_rdk = rp.rdk;
        i_isd = fabs(i_sd) > 1e-3 ? rcp_nr(i_sd) : 0.0;                            // fp.py:792 EPS_S_DOT
        {
          // Horner with running derivatives
          const double t = tp.t;
          const double c0 = pc[5], c1 = pc[6], c2 = pc[7], c3 = pc[8], c4 = pc[9], c5 = pc[10], b3 = pc[11], b4 = pc[12], b5 = pc[13];
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
        R(0, n) = i_rx; R(1, n) = i_ry; R(2, n) = i_cth; R(3, n) = i_sth; R(4, n) = i_rk; R(5, n) = s; R(6, n) = i_isd; R(7, n) = i_sd;
        R(8, n) = A0; R(9, n) = B0; R(10, n) = A1; R(11, n) = B1;
      }
      {
        const bool okp = active && i_rx == i_rx && i_ry == i_ry;
        const unsigned nanm = __ballot_sync(full, active && !okp);                // fp.py:851-866
        if (nanm && fn == 0x7fffffff) fn = n0 + __ffs(nanm) - 1;
        if (has_dyn || M > 0) {
          // box of the pair's reference points (for the obstacle list), fp32 rounded outward
          bxlo = min(bxlo, __reduce_min_sync(full, okp ? f2ord(__double2float_rd(i_rx)) : 0xffffffffu));
          bxhi = max(bxhi, __reduce_max_sync(full, okp ? f2ord(__double2float_ru(i_rx)) : 0u));
          bylo = min(bylo, __reduce_min_sync(full, okp ? f2ord(__double2float_rd(i_ry)) : 0xffffffffu));
          byhi = max(byhi, __reduce_max_sync(full, okp ? f2ord(__double2float_ru(i_ry)) : 0u));
        }
      }
      __syncwarp();                                          // rows of this pass (and of the previous one) are visible

      // ---- phase C: validity chain, lane = sample, loop = lateral targets ----------------------------
      const int keep = fn == 0x7fffffff ? N : (fn >= 2 ? fn : 0);                  // fp.py:866 (final for every sample it excludes)
      const bool valid = active && n < keep;
      const bool chk = valid && n >= 1;                                            // limits skip index 0 (fp.py:964-983)
      const unsigned keep4 = chk ? 0xffffffffu : F_DROP * 0x01010101u;             // n = 0: only the drop guards apply
      // per-item affine coefficients in d_i
      const int np_ = chk ? n - 1 : n;                                            // the previous sample (itself at n = 0)
      const double p_rx = R(0, np_), p_ry = R(1, np_), p_cth = R(2, np_), p_sth = R(3, np_), p_A0 = R(8, np_), p_B0 = R(9, np_);
      const double sd2 = i_sd * i_sd, isd2 = i_isd * i_isd;
      const double Q0 = fma(-i_rk, A0, 1.0), Q1 = -(i_rk * B0);                    // q = 1 - kappa_r d
      const double P0 = A1 * i_isd, P1 = B1 * i_isd;                               // d' (fp.py:792-799)
      const double R0 = (A2 - P0 * i_sdd) * isd2, R1 = (B2 - P1 * i_sdd) * isd2;   // d''
      const double M0 = fma(i_rdk, A0, i_rk * P0), M1 = fma(i_rdk, B0, i_rk * P1); // kappa_r' d + kappa_r d'
      const double S0 = i_sdd * Q0, S1 = i_sdd * Q1;                               // s_ddot q
      // step vector to the previous sample (x = rx - sin d, y = ry + cos d; cc.py:131-132)
      const double E0x = (i_rx - p_rx) - (i_sth * A0 - p_sth * p_A0), E1x = -(i_sth * B0 - p_sth * p_B0);
      const double E0y = (i_ry - p_ry) + (i_cth * A0 - p_cth * p_A0), E1y = i_cth * B0 - p_cth * p_B0;
      const double sd4 = sd2 * sd2;
      unsigned anyslow = 0u;
      // per-item screens for the whole grid of lateral targets (see fot_sweep_items.cuh): `lite` -- no lane needs the
      // road / teleport / speed / singularity / non-finite tests; `skip` -- no lane needs any test
      bool lite, skip;
      {
        const double ga = brake ? 0.0 : P.d_min, gb = brake ? 0.0 : P.d_max, gabs = fmax(fabs(ga), fabs(gb));
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
        lite = __all_sync(full, !valid || lite_ok);                                // NaN anywhere: full chain
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
        skip = __all_sync(full, !valid || (lite_ok && (!chk || ok_rest)));
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
        constexpr bool kLiteLoop = decltype(lite_tag)::value;
#pragma unroll 1
        for (int i0 = 0; i0 < n_dl; i0 += 4) {
          const int left = n_dl - i0;
          const unsigned tailm = left >= 4 ? 0xffffffffu : (1u << (8 * left)) - 1u;
          if (n0 > 0) {
            // a quad whose candidates all carry, from the earlier samples, a flag that outranks everything this loop
            // can still add (fp.py:964-991: drop > speed > acceleration > the rest) is settled
            constexpr unsigned kTop = (kLiteLoop ? (F_DROP | F_SPEED | F_ACCEL) : F_DROP) * 0x01010101u;
            const unsigned t = flags[i0 >> 2] & kTop;
            const unsigned nz = (((t & 0x7f7f7f7fu) + 0x7f7f7f7fu) | t) & 0x80808080u;      // bit 7 of every non-zero byte
            if (((nz | ~tailm) & 0x80808080u) == 0x80808080u) continue;
          }
          unsigned acc = 0u;
          if (valid) {
            // the last quad repeats the last target (its bytes are masked off below): one code path for every grid size
            const int l = n_dl - 1;
            const double g0 = dg[i0], g1 = dg[min(i0 + 1, l)], g2 = dg[min(i0 + 2, l)], g3 = dg[min(i0 + 3, l)];
            sample(lite_tag, g0, acc, 0u); sample(lite_tag, g1, acc, 8u); sample(lite_tag, g2, acc, 16u); sample(lite_tag, g3, acc, 24u);
          }
          const unsigned red = __reduce_or_sync(full, acc & keep4 & tailm);
          if (lane == 0 && red) flags[i0 >> 2] |= red;           // the warp owns the pair: a plain read-modify-write
        }
      };
      if (skip) { }
      else if (lite) sweep_targets(std::true_type{});
      else sweep_targets(std::false_type{});
      // Low-speed regime (fp.py:1022-1032): samples that saw a candidate with v <= 0.5 are listed; the warp
      // redoes the two low-speed tests for them below, one (sample, candidate) unit per lane.
      {
        const unsigned sm = __ballot_sync(full, anyslow && chk);
        if (anyslow && chk) slowq[nslow + __popc(sm & lt_mask)] = (unsigned short)n;
        nslow += __popc(sm);
      }
      // Samples beyond the NaN prefix that are inside the spline domain again still count for the
      // candidate-wide singularity guard (fp.py:826-833 runs before the truncation).  Essentially never.
      __syncwarp();
      if (active && !valid && i_rx == i_rx && keep > 0) {
        for (int i = 0; i < n_dl; ++i) {
          const double qq = fma(dg[i], Q1, Q0);
          if ((qq <= 0.05) & (fabs(qq) < inf)) atomicOr(&flags[i >> 2], F_DROP << (8 * (i & 3)));
        }
      }
      __syncwarp();
    }
    const int keep = fn == 0x7fffffff ? N : (fn >= 2 ? fn : 0);

    // this pair's cost pieces (fot_prepass tables: jerk sums, terminal offset), lane = candidate: issued here, used in phase E
    const int nTv = P.cfg.n_T * B.n_v_max, nTd = P.cfg.n_T * n_d, nB = P.cfg.n_B;
    const double* ct = B.cost_tab + (size_t)q * (nTv + 2 * nTd + 3 * nB);
    const double* ct_s = brake ? ct + nTv + 2 * nTd + kk : ct + jT * B.n_v_max + kk;            // Js
    const double* ct_p = brake ? ct + nTv + 2 * nTd + nB + kk : ct + nTv + jT * n_d;            // Jp[n_dl]
    const double* ct_e = brake ? ct + nTv + 2 * nTd + 2 * nB + kk : ct + nTv + nTd + jT * n_d;  // d_end[n_dl]
    const double e_Js = __ldg(ct_s);
    const double e_Jp = lane < n_dl ? __ldg(ct_p + lane) : 0.0, e_dend = lane < n_dl ? __ldg(ct_e + lane) : 0.0;

    // ---- low-speed tests of unit (listed sample, candidate i): lateral step vs longitudinal step, heading
    // change vs the 0.1 rad / kappa_max * step floor (fp.py:1022-1032), from the item rows
    if (nslow > 0) {
      const int n_su = nslow * n_dl;
      const float rcp_dl = 1.0f / (float)n_dl;
#pragma unroll 1
      for (int u = lane; u < n_su; u += 32) {
        const int ks = __float2int_rz(((float)u + 0.5f) * rcp_dl), i = u - ks * n_dl;
        const int sn = slowq[ks];
        // a candidate that already carries a flag of curvature priority or higher cannot change category
        if ((flags[i >> 2] >> (8 * (i & 3))) & (F_DROP | F_SPEED | F_ACCEL | F_CURV)) continue;
        double r1[kRowW], r0[kRowW];                                             // sample n and sample n - 1 (only checked samples are listed)
#pragma unroll
        for (int f = 0; f < kRowW; ++f) { r1[f] = R(f, sn); r0[f] = R(f, sn - 1); }
        const double di = dg[i];
        const double d = fma(di, r1[9], r1[8]), dprev = fma(di, r0[9], r0[8]);
        const double qq = fma(-r1[4], d, 1.0), dpr = fma(di, r1[11], r1[10]) * r1[6];
        const double ssd = r1[7];
        if (ssd * ssd * fma(qq, qq, dpr * dpr) > 0.25) continue;                 // this candidate is in the fast regime here
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
        if (badc) atomicOr(&flags[i >> 2], F_CURV << (8 * (i & 3)));
      }
      __syncwarp();
    }

    // ---- phase D: collision (fp.py:1035-1233) ----------------------------------------------------------
    const int n_obs = M + SP;
    if (keep > 0 && n_obs > 0 && bxlo != 0xffffffffu) {
      // kinematically clean candidates, lane = candidate: one ballot per word
      int i_lo = -1, i_hi = -1;                            // lowest / highest clean candidate of the pair
#pragma unroll 1
      for (int w = 0; w < G.nwc; ++w) {
        const int ci = 32 * w + lane;
        const unsigned byte = ci < n_dl ? (flags[ci >> 2] >> (8 * (ci & 3))) & 0xffu : 0xffu;
        const unsigned cwd = __ballot_sync(full, byte == 0u);
        if (cwd) { if (i_lo < 0) i_lo = 32 * w + __ffs(cwd) - 1; i_hi = 32 * w + 31 - __clz(cwd); }
        if (lane == 0) cleanw[w] = cwd;
      }
      __syncwarp();
      if (i_lo >= 0) {
        if (!dyn_ready) { mbar_wait(&s_bar, 0u); dyn_ready = true; }
        // the obstacles whose (trajectory) box meets the box of the reference points padded by the widest reach
        // of a clean candidate; a NaN box (fp.py:1211-1222) fails every comparison
        const float bx0 = __fsub_rd(ord2f(bxlo), pad), bx1 = __fadd_ru(ord2f(bxhi), pad);
        const float by0 = __fsub_rd(ord2f(bylo), pad), by1 = __fadd_ru(ord2f(byhi), pad);
        const double ga = d_sorted ? dg[i_lo] : (brake ? 0.0 : P.d_min), gb = d_sorted ? dg[i_hi] : (brake ? 0.0 : P.d_max);
        // One loop, three jobs, whichever is due: (1) list the next obstacles whose box meets the pair's, (2) window
        // test of every kept sample against the listed obstacles, lane = sample, survivors -> queue by ballot + prefix
        // count, (3) exact tests of 32 queued (sample, obstacle) entries, lane = entry, against every live clean candidate.
        int j0 = 0;                                        // next obstacle to list
        int nl = 0, n_st = 0;                              // current list: dynamic entries wl[0, nl), static entries wl[kPairList - n_st, kPairList)
        int c0 = keep;                                     // first sample of the next window pass (>= keep: the list is done)
        unsigned rel_lo = 0u, rel_hi = 0u;                 // this lane's survivors of the last window pass not queued yet: bit e <-> wl[e]
        int pn = 0;                                        // ... and the lane's sample in that pass
        unsigned qh = 0u;                                  // survivor ring: head and
        int qn = 0;                                        //                number of queued entries
        bool finished = false;                             // every obstacle listed, every pass done
        // 32-bit shared-space addresses for the two hot loops (a generic pointer costs the compiler a register pair, or a
        // recomputation from the thread index, per access)
        unsigned wl_a = smem_u32(wl), dg_a = smem_u32(dg), dyn_a = smem_u32(dynst);
        asm volatile("" : "+r"(wl_a), "+r"(dg_a), "+r"(dyn_a));     // opaque: keep them in registers, do not recompute per use
#pragma unroll 1
        for (;;) {
          const unsigned pend = __ballot_sync(full, (rel_lo | rel_hi) != 0u);
          if (pend) {
            // (2b) one survivor of every lane that has any -> queue (ballot + prefix count)
            if (rel_lo | rel_hi) {
              int e;
              if (rel_lo) { e = __ffs(rel_lo) - 1; rel_lo &= rel_lo - 1u; }
              else { e = 32 + __ffs(rel_hi) - 1; rel_hi &= rel_hi - 1u; }
              const unsigned slot = (qh + (unsigned)qn + __popc(pend & lt_mask)) & (kPairQueue - 1);
              q_off[slot] = wl[e];
              q_n[slot] = (unsigned char)pn;
            }
            qn += __popc(pend);
            if (qn < 32) continue;
          } else if (!finished) {
            if (c0 >= keep) {
              if (j0 >= n_obs) { finished = true; continue; }
              // (1) obstacle list, lane = obstacle
              nl = 0; n_st = 0;
#pragma unroll 1
              do {
                const int j = j0 + lane;
                bool in = false;
                unsigned ent = 0u;
                if (j < M) {
                  const double2 o = stat_q[j];
                  in = o.x >= (double)bx0 && o.x <= (double)bx1 && o.y >= (double)by0 && o.y <= (double)by1;
                  ent = 0x80000000u | (unsigned)j;
                } else if (j < n_obs) {
                  const float4 ob = boxes[j - M];                   // xmin xmax ymin ymax
                  in = ob.x <= bx1 && ob.y >= bx0 && ob.z <= by1 && ob.w >= by0;
                  ent = (unsigned)((j - M) * B.T_obs);
                }
                const unsigned m = __ballot_sync(full, in);
                const unsigned ms = j0 >= M ? 0u : (M - j0 >= 32 ? m : m & ((1u << (M - j0)) - 1u));   // the static lanes of this chunk
                if (in) {
                  if (j < M) wl[kPairList - 1 - n_st - __popc(ms & lt_mask)] = ent;
                  else wl[nl + __popc((m & ~ms) & lt_mask)] = ent;
                }
                n_st += __popc(ms);
                nl += __popc(m & ~ms);
                j0 += 32;
              } while (j0 < n_obs && nl + n_st <= kPairList - 32 - 3);
              __syncwarp();
              if (nl > 0 && lane < ((4 - nl) & 3)) wl[nl + lane] = wl[nl - 1];   // pad to a multiple of four (the copies' bits are masked)
              __syncwarp();
              if (nl + n_st > 0) c0 = 0;
              continue;
            }
            // (2a) window test of this pass's samples against the whole list, lane = sample, no votes: a bit per entry.
            // along = (o - ref).t within the collision radius, across = (o - ref).n within the radius of the
            // lateral offsets the pair's clean candidates take at this sample
            const int cn_ = c0 + lane;
            const bool cv = cn_ < keep;
            const int cs_ = cv ? cn_ : 0;
            const double c_rx = R(0, cs_), c_ry = R(1, cs_), cA0 = R(8, cs_), cB0 = R(9, cs_);
            const double c_cth = R(2, cs_), c_sth = R(3, cs_);
            const double nca = -fma(c_rx, c_cth, c_ry * c_sth), ncn = -fma(c_ry, c_cth, -(c_rx * c_sth)), n_sth = -c_sth;
            const double d_lo = cA0 + fmin(ga * cB0, gb * cB0) - 1e-9;
            const double d_hi = cA0 + fmax(ga * cB0, gb * cB0) + 1e-9;
            // a lane beyond the kept samples gets an empty window
            const double w_lo = cv ? d_lo - rc_d : inf, w_hi = d_hi + rc_d;
            const int kob = B.T_obs > 0 ? min(cn_, B.T_obs - 1) : 0;               // clip(round(t/dt)) = n (fp.py:1226-1227)
            auto window = [&](const double2 o) {
              const double al = fma(o.x, c_cth, fma(o.y, c_sth, nca));
              const double ac = fma(o.y, c_cth, fma(o.x, n_sth, ncn));
              return (fabs(al) <= rc_d) & (ac >= w_lo) & (ac <= w_hi);             // NaN -> false
            };
            unsigned lo = 0u, hi = 0u;
            if (stage_dyn) {
              // staged block: four entries per iteration
              unsigned obs_a = dyn_a + 16u * (unsigned)kob;                        // this sample's time step
              asm volatile("" : "+r"(obs_a));
#pragma unroll 1
              for (int e = 0; e < nl; e += 4) {
                unsigned f0, f1, f2, f3;
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(f0), "=r"(f1), "=r"(f2), "=r"(f3) : "r"(wl_a + 4u * (unsigned)e) : "memory");
                double2 o0, o1, o2, o3;
                asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(o0.x), "=d"(o0.y) : "r"(obs_a + 16u * f0) : "memory");
                asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(o1.x), "=d"(o1.y) : "r"(obs_a + 16u * f1) : "memory");
                asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(o2.x), "=d"(o2.y) : "r"(obs_a + 16u * f2) : "memory");
                asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(o3.x), "=d"(o3.y) : "r"(obs_a + 16u * f3) : "memory");
                unsigned nib = 0u;
                if (window(o0)) nib |= 1u;
                if (window(o1)) nib |= 2u;
                if (window(o2)) nib |= 4u;
                if (window(o3)) nib |= 8u;
                if (e < 32) lo |= nib << e; else hi |= nib << (e - 32);
              }
            } else {
              // resident tensor
              const double2* obs_g = dyn_q + kob;
#pragma unroll 1
              for (int e = 0; e < nl; ++e)
                if (window(obs_g[wl[e]])) { if (e < 32) lo |= 1u << e; else hi |= 1u << (e - 32); }
            }
            lo &= nl >= 32 ? 0xffffffffu : (1u << nl) - 1u;                        // the padding's bits
            hi &= nl <= 32 ? 0u : (1u << (nl - 32)) - 1u;
#pragma unroll 1
            for (int k = 0; k < n_st; ++k) {                                       // static entries, from the back of the list
              const int e = kPairList - 1 - k;
              const double2 o = stat_q[wl[e] & 0x7fffffffu];
              const double al = fma(o.x, c_cth, fma(o.y, c_sth, nca));
              const double ac = fma(o.y, c_cth, fma(o.x, n_sth, ncn));
              if (cv & (fabs(al) <= rc_s) & (ac >= d_lo - rc_s) & (ac <= d_hi + rc_s)) { if (e < 32) lo |= 1u << e; else hi |= 1u << (e - 32); }
            }
            rel_lo = lo; rel_hi = hi; pn = cn_;
            c0 += 32;
            continue;
          } else if (qn == 0) {
            break;
          }
          {
            // (3) exact tests of the first min(qn, 32) queued entries: uniform loop over the live clean candidates,
            // one ballot per candidate
            __syncwarp();
            const int cnt = min(qn, 32);
            const bool lv = lane < cnt;
            const unsigned qslot = (qh + (unsigned)lane) & (kPairQueue - 1);
            const unsigned off = lv ? q_off[qslot] : 0u;
            const int en = lv ? (int)q_n[qslot] : 0;
            const bool is_dyn = !(off >> 31);
            const unsigned el = off & 0x7fffffffu;
            double2 o = make_double2(0.0, 0.0);
            if (lv) {
              const unsigned ok_ = el + (unsigned)(B.T_obs > 0 ? min(en, B.T_obs - 1) : 0);
              if (!is_dyn) o = stat_q[el];
              else if (stage_dyn) o = dynst[ok_];
              else o = dyn_q[ok_];
            }
            const double r2 = !lv ? -1.0 : (is_dyn ? r2_dyn : P.cfg.collide_r2);   // idle lanes never hit
            const bool use_budget = budget && is_dyn;
            const double cth = R(2, en), sth = R(3, en), eA0 = R(8, en), eB0 = R(9, en);
            const double X0 = fma(-sth, eA0, R(0, en)) - o.x, X1 = -(sth * eB0);     // x - ox = X0 + d_i X1
            const double Y0 = fma(cth, eA0, R(1, en)) - o.y, Y1 = cth * eB0;
            bool alive = false;
#pragma unroll 1
            for (int w = 0; w < G.nwc; ++w) {
              unsigned live = cleanw[w] & ~hitw[w];
              unsigned nh = 0u;
              if (n_circ == 0 && !budget) {
                // the common case (one circle, decisive hits): nothing but the distance test in the loop
#pragma unroll 1
                while (live) {
                  const int bit = __ffs(live) - 1;
                  live &= live - 1u;
                  double di;
                  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(di) : "r"(dg_a + 8u * (unsigned)(w * 32 + bit)) : "memory");
                  const double dx = fma(di, X1, X0), dy = fma(di, Y1, Y0);
                  if (__ballot_sync(full, dx * dx + dy * dy <= r2)) nh |= 1u << bit;   // fp.py:1196-1198, :1231-1233
                }
              } else {
#pragma unroll 1
                while (live) {
                  const int bit = __ffs(live) - 1;
                  live &= live - 1u;
                  const int i = w * 32 + bit;
                  const double di = dg[i];
                  bool hit = false;
                  if (n_circ == 0) {
                    const double dx = fma(di, X1, X0), dy = fma(di, Y1, Y0);
                    hit = dx * dx + dy * dy <= r2;
                  } else {                                                           // fp.py:1158-1167
                    const double d = fma(di, eB0, eA0);
                    const double dpr = fma(di, R(11, en), R(10, en)) * R(6, en);
                    const double qq = fma(-R(4, en), d, 1.0);
                    const double rh = 1.0 / sqrt(fma(qq, qq, dpr * dpr));
                    const double hx = (cth * qq - sth * dpr) * rh, hy = (sth * qq + cth * dpr) * rh;   // (cos yaw, sin yaw)
                    for (int ci = 0; ci < n_circ && !hit; ++ci) {
                      const double dx = fma(di, X1, X0) + P.cfg.circle_offsets[ci] * hx, dy = fma(di, Y1, Y0) + P.cfg.circle_offsets[ci] * hy;
                      hit = dx * dx + dy * dy <= r2;
                    }
                  }
                  if (use_budget) {
                    if (hit) { const int sidx = (int)(el / (unsigned)B.T_obs) / B.P; atomicOr(&viol[i * vwords + (sidx >> 5)], 1u << (sidx & 31)); }
                    hit = false;
                  }
                  if (__ballot_sync(full, hit)) nh |= 1u << bit;
                }
              }
              if (nh && lane == 0) hitw[w] |= nh;
              alive |= (cleanw[w] & ~(hitw[w] | nh)) != 0u;
            }
            qh += (unsigned)cnt;
            qn -= cnt;
            __syncwarp();
            if (!alive && !budget) break;                  // every clean candidate has its decisive hit
          }
        }
      }
    }

    // ---- phase E: category, cost, arg-min, histogram: lane = candidate ------------------------------
    __syncwarp();
#pragma unroll 1
    for (int c0 = 0; c0 < n_dl; c0 += 32) {
      const int ci = c0 + lane;
      int cat = -1;
      if (ci < n_dl) {
        // cost on the un-truncated profile (fp.py:703-734); jerk sums and terminal offsets from fot_prepass
        const double Jp = c0 == 0 ? e_Jp : __ldg(ct_p + ci), d_end = c0 == 0 ? e_dend : __ldg(ct_e + ci);
        const double Jd = d_end * d_end;
        const double dv = qc[10] - R(7, N - 1);                                   // terminal speed (fp.py:724)
        const double Jv = dv * dv;
        const double Jt = (double)(N - 1) * dt;
        const double lat_cost = P.cfg.k_j * Jp + P.cfg.k_t * Jt + P.cfg.k_d * Jd;
        const double lon_cost = P.cfg.k_j * e_Js + P.cfg.k_t * Jt + P.cfg.k_s_dot * Jv;
        const double cost = P.cfg.k_lat * lat_cost + P.cfg.k_lon * lon_cost;
        const unsigned byte = (flags[ci >> 2] >> (8 * (ci & 3))) & 0xffu;
        if (keep == 0 || (byte & F_DROP)) cat = FOT_CAT_DROP;                     // fp.py:831-833, :933, :944, :953
        else if (byte & F_SPEED) cat = FOT_CAT_SPEED;
        else if (byte & F_ACCEL) cat = FOT_CAT_ACCEL;
        else if (byte & F_CURV) cat = FOT_CAT_CURV;
        else if (byte & F_LAT) cat = FOT_CAT_LAT;
        else if (byte & F_ROAD) cat = FOT_CAT_ROAD;
        else {
          bool hit = (hitw[ci >> 5] >> (ci & 31)) & 1u;
          if (vwords > 0) {
            int nv = 0;
            for (int w = 0; w < vwords; ++w) nv += __popc(viol[ci * vwords + w]);
            hit = hit || nv > max_viol;                                            // fp.py:1113-1124
          }
          if (hit) {
            cat = FOT_CAT_COLL;                                                    // fp.py:986-989
          } else {
            cat = FOT_CAT_OK;
            if (stop_dist == stop_dist) {                                          // fp.py:307-324: v at the last kept sample
              const int kl = keep - 1;
              const double di = dg[ci];
              const double l_rk = R(4, kl), l_isd = R(6, kl), l_sd = R(7, kl);
              const double lQ0 = fma(-l_rk, R(8, kl), 1.0), lQ1 = -(l_rk * R(9, kl));
              const double lP0 = R(10, kl) * l_isd, lP1 = R(11, kl) * l_isd;
              const double qq = fma(di, lQ1, lQ0), dpr = fma(di, lP1, lP0);
              const double v_last = sqrt((l_sd * l_sd) * fma(qq, qq, dpr * dpr));
              const double s_span = R(5, kl) - R(5, 0);
              if (!(v_last <= 0.15 && s_span <= stop_dist + 1e-6)) cat = FOT_CAT_STOP;
            }
          }
        }
        const int cand_idx = cand0 + ci;
        if (O.cand_cat) O.cand_cat[(size_t)q * O.cand_stride + cand_idx] = (uint8_t)cat;
        if (O.cand_cost) O.cand_cost[(size_t)q * O.cand_stride + cand_idx] = cost;
        if (cat == FOT_CAT_OK && cost < INFINITY) argmin_merge(my_cost, my_idx, cost, cand_idx);
      }
      // histogram: the lanes of one category elect a leader, which adds their number to the CTA's counter
      {
        const unsigned peers = __match_any_sync(full, cat);
        if (cat >= 0 && cat < FOT_N_STATS && lane == __ffs(peers) - 1) atomicAdd(&s_stats[cat], __popc(peers));
      }
    }
    __syncwarp();                                          // the slice is free for the next pair
  }  // pairs of this warp

  if (staged && !dyn_ready) mbar_wait(&s_bar, 0u);         // the bulk copy must have landed before the CTA can exit
  for (int off = 16; off > 0; off >>= 1) {
    const double oc = __shfl_down_sync(full, my_cost, off);
    const int oi = __shfl_down_sync(full, my_idx, off);
    argmin_merge(my_cost, my_idx, oc, oi);
  }
  if (lane == 0) { s_cost[wid] = my_cost; s_idx[wid] = my_idx; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < (bd >> 5); ++w) argmin_merge(my_cost, my_idx, s_cost[w], s_idx[w]);
    O.part_cost[part] = my_cost;
    O.part_idx[part] = (my_idx == 0x7fffffff) ? -1 : my_idx;
  }
  if (tid < FOT_N_STATS && s_stats[tid] != 0) atomicAdd(&O.stats[(size_t)q * FOT_N_STATS + tid], s_stats[tid]);
}

}  // namespace fot
