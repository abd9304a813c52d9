// fot_kernels.cuh -- the kernels of the Frenet candidate sweep (sm_100a, fp64).
//
//   fot_obstacle_prepass / fot_static_prepass :
//        reference layout [q][S][P][T][2] -> time-major planes [q][T][3][SPp] of (-2x, -2y, x^2+y^2)
//        (+ the NaN-pedestrian rule, + max |o|^2 per query for the rounding band)
//   fot_sweep  : ONE fused kernel for the whole candidate sweep of every query:
//        coefficient solve -> time-grid evaluation -> spline Frenet->global -> validity chain ->
//        same-time collision test -> cost -> block arg-min.  No trajectory is written to HBM.
//   fot_winner : per query, reduce the block partials and regenerate the 15 sequences of the
//        winning candidate only, in the reference's arithmetic order.
#pragma once
#include "fot_device.cuh"

namespace fot {

constexpr int kSweepThreads = 128;
// Reference-line samples per (terminal speed, t_n), two shared-memory tables:
constexpr int kHot = 4;    // rx ry cos(rtheta) sin(rtheta)            -- both passes
constexpr int kKin = 8;    // rk rdk s sd | sdd 1/sd 1/sd^2 rtheta      -- kinematic pass (+ footprint heading)
constexpr int kRec = 8;    // doubles per compacted collision record: a0..a5, {hold,kl}, {keep,owner}

// flag bits of the priority chain fp.py:964-991
enum : unsigned { F_SPEED = 1u, F_ACCEL = 2u, F_CURV = 4u, F_LAT = 8u, F_ROAD = 16u };

struct SweepGeom {
  int32_t blocks_per_query;  // grid_blocks + brake_blocks
  int32_t grid_blocks;       // ceil(n_T * n_v_max * n_d / ch_eff): the (T, v, d) grid flattened in generation order
  int32_t ch_eff;            // candidates per grid block (<= kSweepThreads)
  int32_t kv_cap;            // terminal speeds (or brake horizons) whose reference samples fit one block
  int32_t brake_blocks;
  int32_t jp_cap;            // max(n_d, kv_cap): per-block lateral-profile slots
  int32_t tile_cap;          // obstacle entries (per plane) one ring stage holds; multiple of 4
  int32_t n_stages;          // ring depth
  int32_t phase2_off;        // offset (doubles) of the ring + record region in dynamic shared memory
  int32_t ints_off;          // offset (doubles) of the int tables
};
constexpr int kMaxStages = 4;
constexpr int kGmax = 8;       // time steps culled / consumed per group
constexpr int kCullCap = 16;   // relevant obstacles listed per (speed, step); more -> full scan of the plane

__device__ __forceinline__ int pad4(int n) { return (n + 3) & ~3; }

__device__ __forceinline__ void atomic_max_pos(double* addr, double v) {   // v >= 0, finite
  atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}

// Per-launch initialisation (kept off the copy engines, which cudaMemsetAsync may use and which are
// busy with the next chunk's upload in the pipelined host path).
__global__ void fot_init_kernel(int32_t* stats, int n_stats, double* max2_a, int n_a, double* max2_b, int n_b,
                                uint8_t* cand_cat, size_t n_cat) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = i; j < (size_t)n_stats; j += stride) stats[j] = 0;
  for (size_t j = i; j < (size_t)n_a; j += stride) max2_a[j] = 0.0;
  for (size_t j = i; j < (size_t)n_b; j += stride) max2_b[j] = 0.0;
  for (size_t j = i; j < n_cat; j += stride) cand_cat[j] = FOT_CAT_DROP + 1;
}

// ----------------------------------------------------------------------------------------
// Obstacle prepass.  One warp per predicted pedestrian trajectory (q, sample, ped).
// The reference drops a pedestrian from a candidate's test when its trajectory AABB misses the
// path AABB (fp.py:1211-1222).  For finite data that prefilter cannot change the result (a sample
// within r of a path point lies inside both padded boxes), but a NaN anywhere in a trajectory
// makes np.min/np.max NaN and so removes that pedestrian entirely; the prepass reproduces
// exactly that by writing NaN for every step of such a trajectory.
// Output per (q, k): three planes of SPp = pad4(S*P) doubles: -2x, -2y, x^2+y^2 (pad: 0, 0, NaN).
// ----------------------------------------------------------------------------------------
__global__ void fot_obstacle_prepass(const double2* __restrict__ dyn, double* __restrict__ tm,
                                     double* __restrict__ max2, int n_q, int SP, int T_obs) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= n_q * SP) return;
  const int q = warp / SP, j = warp % SP;
  const int SPp = pad4(SP);
  const double2* src = dyn + (size_t)warp * T_obs;
  bool bad = false;
  for (int k = lane; k < T_obs; k += 32) {
    const double2 o = src[k];
    bad |= (o.x != o.x) || (o.y != o.y);
  }
  bad = __any_sync(0xffffffffu, bad);
  double* dst = tm + (size_t)q * T_obs * 3 * SPp + j;
  double m2 = 0.0;
  for (int k = lane; k < T_obs; k += 32) {
    const double2 o = src[k];
    double a = -2.0 * o.x, b = -2.0 * o.y, c = o.x * o.x + o.y * o.y;
    if (bad) a = b = c = qnan();
    else if (isfinite(c)) m2 = fmax(m2, c);
    double* row = dst + (size_t)k * 3 * SPp;
    row[0] = a; row[SPp] = b; row[2 * SPp] = c;
    if (j == SP - 1)
      for (int e = SP; e < SPp; ++e) { row[e - j] = 0.0; row[SPp + e - j] = 0.0; row[2 * SPp + e - j] = qnan(); }
  }
  for (int off = 16; off > 0; off >>= 1) m2 = fmax(m2, __shfl_down_sync(0xffffffffu, m2, off));
  if (lane == 0 && m2 > 0.0) atomic_max_pos(max2 + q, m2);
}

// Static obstacles [nq_s][M][2] -> [nq_s][3][Mp].
__global__ void fot_static_prepass(const double2* __restrict__ st, double* __restrict__ out,
                                   double* __restrict__ max2, int nq_s, int M) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq_s * M) return;
  const int q = i / M, j = i % M, Mp = pad4(M);
  const double2 o = st[i];
  const double c = o.x * o.x + o.y * o.y;
  double* row = out + (size_t)q * 3 * Mp + j;
  row[0] = -2.0 * o.x; row[Mp] = -2.0 * o.y; row[2 * Mp] = c;
  if (j == M - 1)
    for (int e = M; e < Mp; ++e) { row[e - j] = 0.0; row[Mp + e - j] = 0.0; row[2 * Mp + e - j] = qnan(); }
  if (isfinite(c) && c > 0.0) atomic_max_pos(max2 + q, c);
}

// ----------------------------------------------------------------------------------------
// Point-vs-obstacle test of one trajectory sample against `cnt` obstacles stored as planes
// A = -2x, B = -2y, C = x^2+y^2 (plane stride `ps`, padded to a multiple of 4).
//   |p - o|^2 = |p|^2 + (px*A + py*B + C): two FMAs and one compare per obstacle.
// The expanded form rounds differently from the reference's (dx*dx + dy*dy), so the compare uses
// a threshold widened by a rigorous rounding band; any sample inside the band ("maybe") is re-tested
// with the reference's exact un-fused expression (fp.py:1196-1198, :1231-1233).  The hit decision
// is therefore identical to NumPy's; the band is ~1e-11 relative, so re-tests are vanishingly rare.
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ bool hits_any(const double* __restrict__ A, int cnt, int ps, double px, double py,
                                         double r2, double omax2) {
  const double pp = fma(px, px, py * py);
  const double band = 3.5527136788005009e-15 * (pp + omax2) + 8.8817841970012523e-16 * r2;   // 2^-48, 2^-50
  const double thr = r2 - pp + band;
  const double* __restrict__ B = A + ps;
  const double* __restrict__ C = B + ps;
  const int cntp = pad4(cnt);
#pragma unroll 2
  for (int j = 0; j < cntp; j += 4) {
    const double2 a01 = *reinterpret_cast<const double2*>(A + j);
    const double2 a23 = *reinterpret_cast<const double2*>(A + j + 2);
    const double2 b01 = *reinterpret_cast<const double2*>(B + j);
    const double2 b23 = *reinterpret_cast<const double2*>(B + j + 2);
    const double2 c01 = *reinterpret_cast<const double2*>(C + j);
    const double2 c23 = *reinterpret_cast<const double2*>(C + j + 2);
    const double t0 = fma(px, a01.x, fma(py, b01.x, c01.x));
    const double t1 = fma(px, a01.y, fma(py, b01.y, c01.y));
    const double t2 = fma(px, a23.x, fma(py, b23.x, c23.x));
    const double t3 = fma(px, a23.y, fma(py, b23.y, c23.y));
    if ((t0 <= thr) | (t1 <= thr) | (t2 <= thr) | (t3 <= thr)) {
      // inside the band: decide with the reference's exact un-fused arithmetic
      const double ax[4] = {a01.x, a01.y, a23.x, a23.y}, bx[4] = {b01.x, b01.y, b23.x, b23.y};
      const double cx[4] = {c01.x, c01.y, c23.x, c23.y};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (cx[e] != cx[e]) continue;         // padding / NaN-trajectory entries never hit
        const double dx = px - (-0.5 * ax[e]), dy = py - (-0.5 * bx[e]);
        if (dx * dx + dy * dy <= r2) return true;
      }
    }
  }
  return false;
}

// Everything the per-candidate passes need that is uniform over a block.
struct BlockCtx {
  const double* tt;     // [NT][kTT]
  const double* hot;    // [kv_cap*NT][kHot]
  const double* kin;    // [kv_cap*NT][kKin]
  const int* kobs;      // [NT] obstacle time index of sample n (fp.py:1226-1227)
  int NT, N;
};

struct KinResult {
  int category;   // FOT_CAT_* decided by the kinematic chain, or -1: clean, collision test needed
  int keep;       // samples kept after the NaN-prefix truncation (fp.py:866)
  double v_last, s_last, s_first;
};

// Pass K: validity chain of one candidate, samples in time order (fp.py:826-833, :851-875, :933-984).
__device__ __forceinline__ KinResult kinematic_pass(const Plan& P, const BlockCtx& C, const Lat& lat, int kl,
                                                    const double* __restrict__ lim) {
  const int N = C.N;
  const double* tt = C.tt;
  const double* hot = C.hot + (size_t)kl * C.NT * kHot;
  const double* kin = C.kin + (size_t)kl * C.NT * kKin;
  const double vmax = lim[0], amax = lim[1], kmax = lim[2], latmax = lim[3];
  const double road_thr = P.cfg.max_road_width + 1e-9;                       // fp.py:982
  const double tele_thr = fmax(vmax, P.cfg.max_speed) * P.cfg.dt * 3.0;      // fp.py:955
  const double tele_thr2 = tele_thr * tele_thr;
  const double kTan01Sq = 0.010067046422495888;                              // tan(0.1)^2

  int first_nan = -1;
  bool singular = false, nonfinite = false;
  double max_step2 = 0.0;
  unsigned flags = 0;
  double x_prev = 0, y_prev = 0, s_prev = 0, d_prev = 0, q_prev = 1, dp_prev = 0;
  KinResult R;
  R.v_last = 0; R.s_last = 0; R.s_first = kin[2];
  const int hold = lat.hold;

  // Straight-line body: every quantity is computed for every sample and the updates are masked by
  // `valid` (sample belongs to the kept prefix), so the loop has no control-flow merges except the
  // rare low-speed regime.  NaN samples beyond the prefix only feed masked updates.
  for (int n = 0; n < N; ++n) {
    const double* h = hot + n * kHot;
    const double* r = kin + n * kKin;
    const double rk = r[0];
    double d, d1, d2;
    lat_fast(lat, tt[kTT * min(n, hold)], d, d1, d2);
    const bool held = n > hold;                                              // fp.py:487-499 brake padding
    d1 = held ? 0.0 : d1;
    d2 = held ? 0.0 : d2;
    const double q1 = fma(-rk, d, 1.0);                                      // fp.py:826-827
    singular |= (q1 <= 0.05) & (fabs(q1) < INFINITY);
    const double x = fma(-h[3], d, h[0]);                                    // cc.py:131
    const double y = fma(h[2], d, h[1]);                                     // cc.py:132
    first_nan = (first_nan < 0 && x != x) ? n : first_nan;                   // fp.py:851-866
    const bool valid = first_nan < 0;
    const double s = r[2], sd = r[3], sdd = r[4];
    const KinPt c = kinematics_fast(rk, r[1], sd, sdd, r[5], r[6], d, d1, d2);
    nonfinite |= valid & !(fabs(c.v) + fabs(c.a) + fabs(c.kappa) < INFINITY);   // fp.py:944-946
    const bool chk = valid & (n >= 1);                                       // limits skip index 0 (fp.py:964-983)
    const double ex = x - x_prev, ey = y - y_prev;
    const double step2 = fma(ex, ex, ey * ey);                               // fp.py:954 (squared)
    max_step2 = (chk & (step2 > max_step2)) ? step2 : max_step2;
    const bool fast = c.v > 0.5;                                             // fp.py:1019
    unsigned f = 0;
    f |= (c.v > vmax) ? F_SPEED : 0u;                                        // fp.py:964
    f |= (fabs(c.a) > amax) ? F_ACCEL : 0u;                                  // fp.py:966
    f |= (fast & (fabs(c.kappa) > kmax)) ? F_CURV : 0u;                      // fp.py:1020
    f |= (c.v * c.v * fabs(c.kappa) > latmax) ? F_LAT : 0u;                  // fp.py:975
    f |= (fabs(d) > road_thr) ? F_ROAD : 0u;                                 // fp.py:982
    flags |= chk ? f : 0u;
    if (chk & !fast & !(flags & F_CURV)) {                                   // fp.py:1022-1032 (rare)
      if (fabs(d - d_prev) > fmax(1.5 * fabs(s - s_prev), 0.02)) {
        flags |= F_CURV;
      } else {
        // |wrap(yaw_i - yaw_{i-1})| is the angle between the heading vectors u = R(rtheta)(q, d').
        const double* hp = h - kHot;
        const double ux = h[2] * c.q - h[3] * c.d_p, uy = h[3] * c.q + h[2] * c.d_p;
        const double ux_prev = hp[2] * q_prev - hp[3] * dp_prev, uy_prev = hp[3] * q_prev + hp[2] * dp_prev;
        const double cr = ux_prev * uy - uy_prev * ux, dt_ = ux_prev * ux + uy_prev * uy;
        if (kmax * kmax * step2 <= 0.01) {
          // threshold is the 0.1 rad floor: angle > 0.1  <=>  dot <= 0 or cross^2 > tan(0.1)^2 dot^2
          if (dt_ <= 0.0 || cr * cr > kTan01Sq * dt_ * dt_) flags |= F_CURV;
        } else if (fabs(atan2(cr, dt_)) > kmax * sqrt(step2)) {
          flags |= F_CURV;
        }
      }
    }
    x_prev = x; y_prev = y; s_prev = s; d_prev = d; q_prev = c.q; dp_prev = c.d_p;
    R.v_last = valid ? c.v : R.v_last;
    R.s_last = valid ? s : R.s_last;
  }

  R.keep = first_nan < 0 ? N : (first_nan >= 2 ? first_nan : 0);            // fp.py:866
  if (singular || R.keep == 0 || nonfinite) R.category = FOT_CAT_DROP;       // fp.py:831-833, :933, :944
  else if (R.keep >= 2 && max_step2 > tele_thr2) R.category = FOT_CAT_DROP;  // fp.py:953-956
  else if (flags & F_SPEED) R.category = FOT_CAT_SPEED;
  else if (flags & F_ACCEL) R.category = FOT_CAT_ACCEL;
  else if (flags & F_CURV) R.category = FOT_CAT_CURV;
  else if (flags & F_LAT) R.category = FOT_CAT_LAT;
  else if (flags & F_ROAD) R.category = FOT_CAT_ROAD;
  else R.category = -1;
  return R;
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

// One obstacle tile of the collision pass: `n_planes` time planes (small fields: several whole
// planes per tile) or one chunk of one plane (large fields).  Entries of a plane are stored in the
// stage as [A | B | C] with plane stride 3*cnt.
struct Tile {
  int k0, n_planes, e0, cnt;   // first time plane, planes in the tile, first entry, entries per plane (multiple of 4)
};
struct TilePlan {
  int SPp, cap, planes_per_tile, chunks_per_plane, n_tiles, K_used;
  __device__ __forceinline__ void init(int SPp_, int cap_, int K_used_) {
    SPp = SPp_; cap = cap_; K_used = K_used_;
    if (SPp <= cap) { planes_per_tile = cap / SPp; chunks_per_plane = 1; n_tiles = (K_used + planes_per_tile - 1) / planes_per_tile; }
    else { planes_per_tile = 1; chunks_per_plane = (SPp + cap - 1) / cap; n_tiles = K_used * chunks_per_plane; }
  }
  __device__ __forceinline__ Tile tile(int t) const {
    Tile T;
    if (chunks_per_plane == 1) { T.k0 = t * planes_per_tile; T.n_planes = min(planes_per_tile, K_used - T.k0); T.e0 = 0; T.cnt = SPp; }
    else { T.k0 = t / chunks_per_plane; T.n_planes = 1; T.e0 = (t % chunks_per_plane) * cap; T.cnt = min(cap, SPp - T.e0); }
    return T;
  }
};

// Issue the bulk copies of tile `T` of `planes` ([K][3][SPp] doubles) into `stage`.
__device__ __forceinline__ void tile_issue(const double* planes, const TilePlan& TP, const Tile& T, double* stage, uint64_t* bar) {
  const uint32_t bytes = (uint32_t)T.n_planes * 3u * (uint32_t)T.cnt * 8u;
  mbar_expect_tx(bar, bytes);
  if (TP.chunks_per_plane == 1) {
    tma_bulk_g2s(stage, planes + (size_t)T.k0 * 3 * TP.SPp, bytes, bar);
  } else {
    const double* src = planes + (size_t)T.k0 * 3 * TP.SPp + T.e0;
    for (int pl = 0; pl < 3; ++pl) tma_bulk_g2s(stage + pl * T.cnt, src + (size_t)pl * TP.SPp, (uint32_t)T.cnt * 8u, bar);
  }
}

// Per-thread state of the collision pass.
struct CollState {
  bool live;        // still needs testing (kinematically clean, no decisive hit yet)
  bool hit;
  int keep, kl;
};

// Test sample n of this thread's candidate against one staged plane (cnt entries at A).
__device__ __forceinline__ bool sample_hits(const Plan& P, const BlockCtx& C, const Lat& lat, int kl, int n,
                                            const double* A, int cnt, double r2, double omax2) {
  const double* h = C.hot + ((size_t)kl * C.NT + n) * kHot;
  const double d = lat_fast0(lat, C.tt[kTT * (n > lat.hold ? lat.hold : n)]);
  const double x = fma(-h[3], d, h[0]);
  const double y = fma(h[2], d, h[1]);
  const int n_circ = P.cfg.n_circles;
  if (n_circ == 0) return hits_any(A, cnt, cnt, x, y, r2, omax2);
  const double* r = C.kin + ((size_t)kl * C.NT + n) * kKin;                    // (not aliased in footprint mode)
  const double d_p = lat_p1(lat, C.tt, n) * r[5];                              // fp.py:1158-1167
  const double yaw = wrap_angle(atan2(d_p, 1.0 - r[0] * d) + r[7]);
  double hx, hy;
  sincos(yaw, &hy, &hx);
  for (int ci = 0; ci < n_circ; ++ci)
    if (hits_any(A, cnt, cnt, x + P.cfg.circle_offsets[ci] * hx, y + P.cfg.circle_offsets[ci] * hy, r2, omax2)) return true;
  return false;
}

// Chance-constrained variant with a violation budget (fp.py:1113-1124): rare mode, straight from
// global memory, exact arithmetic, per-sample early-out.
__device__ __forceinline__ bool collision_budget(const Plan& P, const Batch& B, const BlockCtx& C, int q,
                                                 const Lat& lat, int kl, int keep, int max_viol) {
  const int SP = B.S * B.P, SPp = pad4(SP);
  const double* obs_q = B.obs_tm + (size_t)q * B.T_obs * 3 * SPp;
  const double r2 = P.cfg.collide_r2;
  const int n_circ = P.cfg.n_circles;
  unsigned long long viol = 0ull;
  for (int n = 0; n < keep; ++n) {
    const double* h = C.hot + ((size_t)kl * C.NT + n) * kHot;
    const double* r = C.kin + ((size_t)kl * C.NT + n) * kKin;
    const double d = lat_fast0(lat, C.tt[kTT * (n > lat.hold ? lat.hold : n)]);
    const double x = fma(-h[3], d, h[0]), y = fma(h[2], d, h[1]);
    double hx = 0.0, hy = 0.0;
    if (n_circ > 0) {
      const double d_p = lat_p1(lat, C.tt, n) * r[5];
      const double yaw = wrap_angle(atan2(d_p, 1.0 - r[0] * d) + r[7]);
      sincos(yaw, &hy, &hx);
    }
    const double* ob = obs_q + (size_t)C.kobs[n] * 3 * SPp;
    for (int ci = 0; ci < (n_circ > 0 ? n_circ : 1); ++ci) {
      const double px = n_circ > 0 ? x + P.cfg.circle_offsets[ci] * hx : x;
      const double py = n_circ > 0 ? y + P.cfg.circle_offsets[ci] * hy : y;
      for (int sidx = 0; sidx < B.S; ++sidx) {
        if ((viol >> sidx) & 1ull) continue;
        bool hit = false;
        for (int p = sidx * B.P; p < (sidx + 1) * B.P && !hit; ++p) {
          const double dx = px - (-0.5 * ob[p]), dy = py - (-0.5 * ob[SPp + p]);
          hit = dx * dx + dy * dy <= r2;
        }
        if (hit) viol |= (1ull << sidx);
      }
      if (__popcll(viol) > max_viol) return true;
    }
  }
  return false;
}

// ----------------------------------------------------------------------------------------
// The sweep kernel.  Block b of query q covers either `ch_eff` consecutive (v, d) candidates of
// one horizon T_j, or up to `kv_cap` brake-ladder candidates.
//   phase 0: time-power table; quartic solve + jerk sum per terminal speed; lateral jerk sums;
//            reference-line samples (s(t), spline, heading, curvature) per (speed, t_n) -> smem
//   phase 1: one thread per candidate: cost + kinematic validity chain
//   phase 2: collision test of the kinematically clean candidates, the block in lockstep over
//            obstacle tiles that one thread streams into a shared-memory ring with TMA bulk
//            copies (cp.async.bulk + mbarrier), static obstacles first, then the time planes
//   phase 3: stop-distance filter, block arg-min by (cost, index), category histogram
// ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kSweepThreads, 5)
fot_sweep(const Plan P, const Batch B, const Out O, const SweepGeom G) {
  extern __shared__ double sm[];
  const int NT = P.n_t_max;
  double* tt = sm;                                         // [NT][kTT]
  double* hot = tt + kTT * NT;                             // [kv_cap*NT][kHot]
  double* js = hot + (size_t)kHot * G.kv_cap * NT;         // [kv_cap]
  double* lonc = js + G.kv_cap;                            // [5][kv_cap]
  double* jp = lonc + 5 * G.kv_cap;                        // [jp_cap] lateral jerk sums
  double* dend = jp + G.jp_cap;                            // [jp_cap] terminal lateral offsets
  double* kin = dend + G.jp_cap;                           // [kv_cap*NT][kKin]
  // phase-2 region: obstacle ring + compacted records.  When it fits (and no footprint needs the
  // kinematic table in phase 2) it re-uses the kinematic table's memory, which is dead by then.
  double* ring = sm + G.phase2_off;                        // [n_stages][3*tile_cap] obstacle tiles (16 B aligned)
  double* rec = ring + (size_t)G.n_stages * 3 * G.tile_cap;   // [kSweepThreads][kRec]
  int* holdk = reinterpret_cast<int*>(sm + G.ints_off);    // [kv_cap]
  int* kobs = holdk + G.kv_cap;                            // [NT]
  int* hitf = kobs + NT;                                   // [kSweepThreads] collision verdict per owner thread
  int* pair_live = hitf + kSweepThreads;                   // [kv_cap] any clean candidate with this profile?
  int* pairN = pair_live + G.kv_cap;                       // [kv_cap] samples of the pair's profile
  int* pairT = pairN + G.kv_cap;                           // [kv_cap] horizon index (or brake horizon index)
  int* ccnt = pairT + G.kv_cap;                        // [kv_cap*kGmax] relevant obstacles per (speed, step)
  unsigned short* clist = reinterpret_cast<unsigned short*>(ccnt + G.kv_cap * kGmax);   // [kv_cap*kGmax][kCullCap]
  __shared__ int s_wcnt[kSweepThreads / 32];
  __shared__ int s_Nmax;
  __shared__ int s_stats[FOT_N_STATS];
  __shared__ double s_cost[kSweepThreads / 32];
  __shared__ int s_idx[kSweepThreads / 32];
  __shared__ __align__(8) uint64_t s_bar[kMaxStages];

  const int q = blockIdx.x / G.blocks_per_query;
  const int b = blockIdx.x % G.blocks_per_query;
  const int tid = threadIdx.x;
  const double* fs = B.frenet + 6 * (size_t)q;
  const int n_v = B.n_v[q];
  const int n_d = P.cfg.n_d;
  const int n_grid_blocks = G.grid_blocks;
  const bool brake_blk = b >= n_grid_blocks;
  const size_t part = (size_t)q * G.blocks_per_query + b;

  // A "pair" is one longitudinal profile: (horizon T_j, terminal speed v_k) of the grid, or one brake
  // horizon.  The grid's candidates are flattened in generation order m = (j_T*n_v + k_v)*n_d + i_d
  // and cut into blocks of ch_eff, so every thread of every block but the last owns a candidate; a
  // block therefore spans a few pairs, possibly of two horizons (different sample counts).
  int m0 = 0, k_lo = 0, n_k = 0, n_cand = 0;
  if (!brake_blk) {
    m0 = b * G.ch_eff;
    const int total = P.cfg.n_T * n_v * n_d;
    if (m0 < total) {
      n_cand = min(G.ch_eff, total - m0);
      k_lo = m0 / n_d;
      n_k = (m0 + n_cand - 1) / n_d - k_lo + 1;
    }
  } else {
    const int b0 = (b - n_grid_blocks) * G.kv_cap;
    if (fs[1] > 0.1 && b0 < P.cfg.n_B) {               // fp.py:469 BRAKE_MIN_SPEED
      k_lo = b0;
      n_k = min(G.kv_cap, P.cfg.n_B - b0);
      n_cand = n_k;
    }
  }
  if (n_cand == 0) {                                   // uniform per block
    if (tid == 0) { O.part_cost[part] = INFINITY; O.part_idx[part] = -1; }
    return;
  }

  // ---- phase 0 ---------------------------------------------------------------------------
  if (tid < FOT_N_STATS) s_stats[tid] = 0;
  if (tid == 0) {
    for (int i = 0; i < G.n_stages; ++i) mbar_init(&s_bar[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int n = tid; n < NT; n += kSweepThreads) {
    tt_fill(tt, n, P.cfg.dt);
    const double kf = rint(((double)n * P.cfg.dt) / P.cfg.dt);               // fp.py:1226-1227
    const int kmax_i = B.T_obs > 0 ? B.T_obs - 1 : 0;
    kobs[n] = kf < 0.0 ? 0 : (kf > (double)kmax_i ? kmax_i : (int)kf);
  }
  if (tid == 0) s_Nmax = 0;
  __syncthreads();
  const int jT_lo = brake_blk ? 0 : k_lo / n_v;
  if (tid < n_k) {
    Lon L;
    int Nk;
    if (!brake_blk) {
      const int p = k_lo + tid, jT = p / n_v, kv = p - jT * n_v;
      Nk = P.n_steps[jT] + 1;
      L = lon_solve(fs, B.v_grid[(size_t)q * B.n_v_max + kv], P.T[jT], P.inv4 + 4 * jT, n_v == 1, Nk - 1);
      pairT[tid] = jT;
    } else {
      Nk = P.cfg.n_total;
      L = lon_solve(fs, 0.0, P.Tb[k_lo + tid], P.inv4b + 4 * (k_lo + tid), true, P.n_steps_b[k_lo + tid]);
      pairT[tid] = k_lo + tid;
    }
    pairN[tid] = Nk;
    atomicMax(&s_Nmax, Nk);
    lonc[tid] = L.a0; lonc[G.kv_cap + tid] = L.a1; lonc[2 * G.kv_cap + tid] = L.a2;
    lonc[3 * G.kv_cap + tid] = L.a3; lonc[4 * G.kv_cap + tid] = L.a4;
    holdk[tid] = L.hold;
    auto jerk2 = [&](int n) { const double j = lon_p3(L, tt, n); return j * j; };
    js[tid] = np_pairwise_sum(jerk2, 0, Nk);            // fp.py:722
  }
  // lateral jerk sum and terminal offset once per lateral profile of this block (fp.py:718-719):
  // slot (j_T - jT_lo) * n_d + i_d for the grid, the brake horizon's index for the ladder
  const int n_Tl = brake_blk ? 0 : (k_lo + n_k - 1) / n_v - jT_lo + 1;
  for (int i = tid; i < (brake_blk ? n_k : n_Tl * n_d); i += kSweepThreads) {
    Lat L;
    int Nl;
    if (brake_blk) {
      Nl = P.cfg.n_total;
      L = lat_solve(fs, fs[3], P.Tb[k_lo + i], P.inv5b + 9 * (k_lo + i), true, P.n_steps_b[k_lo + i]);
    } else {
      const int jT = jT_lo + i / n_d, id = i % n_d;
      Nl = P.n_steps[jT] + 1;
      L = lat_solve(fs, P.d_grid[id], P.T[jT], P.inv5 + 9 * jT, n_d == 1, Nl - 1);
    }
    auto jerk2 = [&](int n) { const double j = lat_p3(L, tt, n); return j * j; };
    jp[i] = np_pairwise_sum(jerk2, 0, Nl);
    dend[i] = lat_p0(L, tt, Nl - 1);
  }
  __syncthreads();
  const int N = s_Nmax;                                 // longest profile in the block
  for (int idx = tid; idx < n_k * N; idx += kSweepThreads) {
    const int kl = idx / N, n = idx - kl * N;
    if (n >= pairN[kl]) continue;
    Lon L;
    L.a0 = lonc[kl]; L.a1 = lonc[G.kv_cap + kl]; L.a2 = lonc[2 * G.kv_cap + kl];
    L.a3 = lonc[3 * G.kv_cap + kl]; L.a4 = lonc[4 * G.kv_cap + kl]; L.hold = holdk[kl];
    const double s = lon_p0(L, tt, n);
    const double sd = lon_p1(L, tt, n);
    const RefPt rp = spline_ref(P, s);
    double sn, cs;
    sincos(rp.rth, &sn, &cs);                           // cc.py:128-129
    const bool moving = fabs(sd) > 1e-3;                // fp.py:792
    const double inv_sd = moving ? 1.0 / sd : 0.0;
    double* h = hot + ((size_t)kl * NT + n) * kHot;
    double* r = kin + ((size_t)kl * NT + n) * kKin;
    h[0] = rp.rx; h[1] = rp.ry; h[2] = cs; h[3] = sn;
    r[0] = rp.rk; r[1] = rp.rdk; r[2] = s; r[3] = sd;
    r[4] = lon_p2(L, tt, n); r[5] = inv_sd; r[6] = inv_sd * inv_sd; r[7] = rp.rth;
  }
  __syncthreads();

  // ---- phase 1: cost + kinematic chain ----------------------------------------------------
  BlockCtx C{tt, hot, kin, kobs, NT, N};
  int kl = 0, cand_idx = 0, cat = FOT_CAT_DROP + 1;     // idle threads: no category
  double cost = INFINITY;
  Lat lat{};
  KinResult K{};
  CollState cs{false, false, 0, 0};
  if (tid < n_cand) {
    int li, Nc;
    if (!brake_blk) {
      const int m = m0 + tid;
      const int p = m / n_d, id = m - p * n_d;
      kl = p - k_lo;
      const int jT = pairT[kl];
      Nc = pairN[kl];
      li = (jT - jT_lo) * n_d + id;
      cand_idx = m;                                      // generation order (fp.py:398-449)
      lat = lat_solve(fs, P.d_grid[id], P.T[jT], P.inv5 + 9 * jT, n_d == 1, Nc - 1);
    } else {
      kl = tid;
      li = tid;
      Nc = P.cfg.n_total;
      cand_idx = P.cfg.n_T * n_v * n_d + k_lo + tid;
      lat = lat_solve(fs, fs[3], P.Tb[k_lo + tid], P.inv5b + 9 * (k_lo + tid), true, P.n_steps_b[k_lo + tid]);
    }
    // cost on the un-truncated profile (fp.py:703-734)
    const double Jp = jp[li];
    const double d_end = dend[li];
    const double Jd = d_end * d_end;
    const double Js = js[kl];
    const double dv = B.target[q] - kin[((size_t)kl * NT + (Nc - 1)) * kKin + 3];
    const double Jv = dv * dv;
    const double Jt = tt[kTT * (Nc - 1)];
    const double lat_cost = P.cfg.k_j * Jp + P.cfg.k_t * Jt + P.cfg.k_d * Jd;
    const double lon_cost = P.cfg.k_j * Js + P.cfg.k_t * Jt + P.cfg.k_s_dot * Jv;
    cost = P.cfg.k_lat * lat_cost + P.cfg.k_lon * lon_cost;
    C.N = Nc;
    K = kinematic_pass(P, C, lat, kl, B.limits + 4 * (size_t)q);
    C.N = N;
    cat = K.category;
    cs.live = cat < 0;
    cs.keep = K.keep;
    cs.kl = kl;
  }

  // ---- phase 2: collision test (fp.py:1035-1233) -------------------------------------------
  const bool dist_mode = (B.dyn_mode == FOT_DYN_DISTRIBUTION);
  const int max_viol = dist_mode ? (int)floor(P.cfg.chance_epsilon * (double)B.S) : 0;   // fp.py:1114
  const int qs = B.static_per_query ? q : 0;
  uint32_t n_issued = 0, n_waited = 0;                  // running tile counters -> stage + parity
  const int n_circ = P.cfg.n_circles;
  double max_off = 0.0;                                 // footprint circles sit within max|offset| of the path point
  for (int i = 0; i < n_circ; ++i) max_off = fmax(max_off, fabs(P.cfg.circle_offsets[i]));
  auto run_tiles = [&](const double* planes, int SPp_, int K_used, bool is_static, double r2, double omax2) {
    TilePlan TP;
    TP.init(SPp_, G.tile_cap, K_used);
    // prologue: fill the ring
    int t_issue = 0;                                    // counters are uniform; only thread 0 issues
    for (; t_issue < min(G.n_stages - 1, TP.n_tiles); ++t_issue, ++n_issued) {
      const int st = n_issued % G.n_stages;
      if (tid == 0) tile_issue(planes, TP, TP.tile(t_issue), ring + (size_t)st * 3 * G.tile_cap, &s_bar[st]);
    }
    for (int t = 0; t < TP.n_tiles; ++t) {
      if (t_issue < TP.n_tiles) {                       // refill the stage freed by the previous barrier
        const int st = n_issued % G.n_stages;
        if (tid == 0) tile_issue(planes, TP, TP.tile(t_issue), ring + (size_t)st * 3 * G.tile_cap, &s_bar[st]);
        ++t_issue; ++n_issued;
      }
      const int st = n_waited % G.n_stages;
      mbar_wait(&s_bar[st], (n_waited / G.n_stages) & 1u);
      ++n_waited;
      // A clean candidate's sample n lies on the normal of the reference line through the
      // (speed, n) reference point, at lateral offset |d| <= wc - rc (road-bound check passed; n = 0
      // is the ego's own offset).  So only obstacles within rc along the tangent and wc across it
      // can touch any candidate of that speed at that step: the block first lists those (a handful
      // out of the whole plane), then every candidate tests its own point against the short list
      // with the reference's exact arithmetic.  Conservative margins make the list a superset.
      const Tile T = TP.tile(t);
      const double* stage = ring + (size_t)st * 3 * G.tile_cap;
      const int n_lo = is_static ? 0 : T.k0;
      const int n_hi = is_static ? N : ((T.k0 + T.n_planes >= K_used) ? N : T.k0 + T.n_planes);
      const double rc = sqrt(r2) * (1.0 + 1e-9) + 1e-9 + max_off;
      const double wc = fmax(P.cfg.max_road_width + 1e-9, fabs(fs[3])) + rc;
      const int lane = tid & 31, warp = tid >> 5;
      bool done = false;
      for (int g0 = n_lo; g0 < n_hi; g0 += kGmax) {
        const int ng = min(kGmax, n_hi - g0);
        for (int pg = warp; pg < n_k * ng; pg += kSweepThreads / 32) {       // cull: one warp per (speed, step)
          const int klc = pg / ng, n = g0 + (pg - klc * ng);
          int total = 0;
          if (pair_live[klc] && n < pairN[klc]) {
            const double* h = hot + ((size_t)klc * NT + n) * kHot;
            const double rx = h[0], ry = h[1], cth = h[2], sth = h[3];
            const double* A = stage + (is_static ? 0 : (size_t)(kobs[n] - T.k0) * 3 * T.cnt);
            for (int j0 = 0; j0 < T.cnt; j0 += 32) {
              const int j = j0 + lane;
              bool rel = false;
              if (j < T.cnt) {
                const double ex = -0.5 * A[j] - rx, ey = -0.5 * A[T.cnt + j] - ry;
                const double cc = A[2 * T.cnt + j];                          // NaN marks padding entries
                rel = fabs(ex * cth + ey * sth) <= rc && fabs(ey * cth - ex * sth) <= wc && cc == cc;   // NaN -> false
              }
              const unsigned m = __ballot_sync(0xffffffffu, rel);
              if (rel) {
                const int pos = total + __popc(m & ((1u << lane) - 1u));
                if (pos < kCullCap) clist[pg * kCullCap + pos] = (unsigned short)j;
              }
              total += __popc(m);
            }
          }
          if (lane == 0) ccnt[pg] = total;
        }
        __syncthreads();
        if (cs.live) {                                                       // consume
          for (int n = g0; n < min(g0 + ng, cs.keep) && !cs.hit; ++n) {
            const int pg = kl * ng + (n - g0);
            const int c = ccnt[pg];
            if (c == 0) continue;
            const double* A = stage + (is_static ? 0 : (size_t)(kobs[n] - T.k0) * 3 * T.cnt);
            if (c > kCullCap || T.cnt > 65535) {                             // list overflow: scan the plane
              cs.hit = sample_hits(P, C, lat, kl, n, A, T.cnt, r2, omax2);
              continue;
            }
            const double* h = hot + ((size_t)kl * NT + n) * kHot;
            const double d = lat_fast0(lat, tt[kTT * (n > lat.hold ? lat.hold : n)]);
            const double x = fma(-h[3], d, h[0]), y = fma(h[2], d, h[1]);
            double hx = 0.0, hy = 0.0;
            if (n_circ > 0) {                                                // fp.py:1158-1167
              const double* r = kin + ((size_t)kl * NT + n) * kKin;
              const double d_p = lat_p1(lat, tt, n) * r[5];
              sincos(wrap_angle(atan2(d_p, 1.0 - r[0] * d) + r[7]), &hy, &hx);
            }
            for (int ci = 0; ci < (n_circ > 0 ? n_circ : 1) && !cs.hit; ++ci) {
              const double px = n_circ > 0 ? x + P.cfg.circle_offsets[ci] * hx : x;
              const double py = n_circ > 0 ? y + P.cfg.circle_offsets[ci] * hy : y;
              for (int e = 0; e < c; ++e) {
                const int j = clist[pg * kCullCap + e];
                const double dx = px - (-0.5 * A[j]), dy = py - (-0.5 * A[T.cnt + j]);
                if (dx * dx + dy * dy <= r2) { cs.hit = true; break; }       // fp.py:1196-1198, :1231-1233
              }
            }
          }
          if (cs.hit) cs.live = false;
        }
        // all reads of the lists / this stage are done; leave early once nobody is live
        if (!__syncthreads_or(cs.live ? 1 : 0)) { done = true; break; }
      }
      if (done) {
        // drain copies already in flight so the ring can be reused / the block can exit
        for (; n_waited < n_issued; ++n_waited) mbar_wait(&s_bar[n_waited % G.n_stages], (n_waited / G.n_stages) & 1u);
        break;
      }
    }
    __syncthreads();
  };
  // Compact the kinematically clean candidates to the low threads so the collision pass runs in
  // dense warps; each record remembers its owner thread, which gets the verdict back through hitf.
  hitf[tid] = 0;
  if (tid < G.kv_cap) pair_live[tid] = 0;
  const unsigned live_mask = __ballot_sync(0xffffffffu, cs.live);
  if ((tid & 31) == 0) s_wcnt[tid >> 5] = __popc(live_mask);
  __syncthreads();                                       // also: every read of `kin` is done
  int n_live = 0, slot = __popc(live_mask & ((1u << (tid & 31)) - 1u));
  for (int w = 0; w < kSweepThreads / 32; ++w) {
    if (w < (tid >> 5)) slot += s_wcnt[w];
    n_live += s_wcnt[w];
  }
  if (n_live > 0) {
    if (cs.live) {
      double* rc = rec + (size_t)slot * kRec;
      rc[0] = lat.a0; rc[1] = lat.a1; rc[2] = lat.a2; rc[3] = lat.a3; rc[4] = lat.a4; rc[5] = lat.a5;
      reinterpret_cast<int*>(rc + 6)[0] = lat.hold; reinterpret_cast<int*>(rc + 6)[1] = kl;
      reinterpret_cast<int*>(rc + 7)[0] = cs.keep;  reinterpret_cast<int*>(rc + 7)[1] = tid;
      pair_live[kl] = 1;
    }
    __syncthreads();
    int owner = 0;
    cs.live = tid < n_live;
    cs.hit = false;
    if (cs.live) {
      const double* rc = rec + (size_t)tid * kRec;
      lat.a0 = rc[0]; lat.a1 = rc[1]; lat.a2 = rc[2]; lat.a3 = rc[3]; lat.a4 = rc[4]; lat.a5 = rc[5];
      lat.hold = reinterpret_cast<const int*>(rc + 6)[0]; kl = reinterpret_cast<const int*>(rc + 6)[1];
      cs.keep = reinterpret_cast<const int*>(rc + 7)[0];  owner = reinterpret_cast<const int*>(rc + 7)[1];
    }
    if (B.static_tm)
      run_tiles(B.static_tm + (size_t)qs * 3 * pad4(B.n_static), pad4(B.n_static), 1, true, P.cfg.collide_r2,
                B.static_max2[qs]);
    if (B.obs_tm) {
      const int SPp = pad4(B.S * B.P);
      if (max_viol == 0) {
        run_tiles(B.obs_tm + (size_t)q * B.T_obs * 3 * SPp, SPp, kobs[N - 1] + 1, false,
                  dist_mode ? P.cfg.collide_r2 : P.cfg.collide_r2_single, B.obs_max2[q]);   // fp.py:1099-1104
      } else if (cs.live) {
        cs.hit = collision_budget(P, B, C, q, lat, kl, cs.keep, max_viol);
      }
    }
    if (cs.hit) hitf[owner] = 1;
    __syncthreads();
  }

  // ---- phase 3 ---------------------------------------------------------------------------
  double my_cost = INFINITY;
  int my_idx = 0x7fffffff;
  if (tid < n_cand) {
    if (cat < 0) {
      if (hitf[tid]) {
        cat = FOT_CAT_COLL;                                                  // fp.py:986-989
      } else {
        cat = FOT_CAT_OK;
        const double stop_dist = B.stop_dist[q];
        if (stop_dist == stop_dist) {                                        // fp.py:307-324
          const bool stops = fabs(K.v_last) <= 0.15;
          if (!(stops && (K.s_last - K.s_first) <= stop_dist + 1e-6)) cat = FOT_CAT_STOP;
        }
      }
    }
    if (cat < FOT_N_STATS) atomicAdd(&s_stats[cat], 1);
    if (O.cand_cat) O.cand_cat[(size_t)q * O.cand_stride + cand_idx] = (uint8_t)cat;
    if (O.cand_cost) O.cand_cost[(size_t)q * O.cand_stride + cand_idx] = cost;
    if (cat == FOT_CAT_OK && cost < INFINITY) { my_cost = cost; my_idx = cand_idx; }
  }
  for (int off = 16; off > 0; off >>= 1) {
    const double oc = __shfl_down_sync(0xffffffffu, my_cost, off);
    const int oi = __shfl_down_sync(0xffffffffu, my_idx, off);
    argmin_merge(my_cost, my_idx, oc, oi);
  }
  if ((tid & 31) == 0) { s_cost[tid >> 5] = my_cost; s_idx[tid >> 5] = my_idx; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < kSweepThreads / 32; ++w) argmin_merge(my_cost, my_idx, s_cost[w], s_idx[w]);
    O.part_cost[part] = my_cost;
    O.part_idx[part] = (my_idx == 0x7fffffff) ? -1 : my_idx;
  }
  if (tid < FOT_N_STATS && s_stats[tid] != 0) atomicAdd(&O.stats[(size_t)q * FOT_N_STATS + tid], s_stats[tid]);
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
fot_winner(const Plan P, const Batch B, const Out O, const SweepGeom G) {
  extern __shared__ double sm[];
  const int NT = P.n_t_max;
  double* tt = sm;   // [NT][kTT]
  __shared__ double s_cost[4];
  __shared__ int s_idx[4];
  __shared__ int s_first_nan;
  const int q = blockIdx.x, tid = threadIdx.x;

  double c = INFINITY;
  int i = 0x7fffffff;
  for (int p = tid; p < G.blocks_per_query; p += blockDim.x) {
    const int pi = O.part_idx[(size_t)q * G.blocks_per_query + p];
    if (pi >= 0) argmin_merge(c, i, O.part_cost[(size_t)q * G.blocks_per_query + p], pi);
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
  if (i == 0x7fffffff) {
    if (tid == 0) {
      O.best_idx[q] = -1; O.best_cost[q] = INFINITY; O.winner_len[q] = 0;
      if (O.m_best_idx) { O.m_best_idx[q] = -1; O.m_best_cost[q] = INFINITY; O.m_winner_len[q] = 0; }
    }
    return;
  }
  const int len = regenerate(P, B, q, i, tt, W, MW, &s_first_nan);
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
