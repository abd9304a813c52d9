// fot_sweep_math.cuh -- what the two sweep kernels share (sm_100a, fp64).
//
// fot_sweep_items (fot_sweep_items.cuh) and fot_sweep_pairs (fot_sweep_pairs.cuh) cut the work differently -- blocks of
// pairs with block barriers against one pair per warp -- and call the same functions for the pieces below: the wait for
// the gated upload slice, the boxes of a staged obstacle block, the reference point over either table layout (as an
// accessor, so that the pair kernel's compile-time strides stay compile-time), and the validity chain's flag idiom.
//
// The per-candidate arithmetic of the validity chain, the low-speed and collision tests, the category chain and the cost
// is still written out in each kernel (DESIGN.md section 3 says why): both kernels are tuned to the instruction, and
// every sharing of those pieces tried so far changed the SASS ptxas emits for one of them.
//
// Reference citations: fp.py = src/planning/frenet_planner.py, cs.py = cubic_spline.py,
// cc.py = src/core/coordinate_converter.py.
#pragma once
#include "fot_kernels.cuh"

namespace fot {

constexpr int kRowW = 12;           // item row: rx ry cos sin | kappa s 1/s_dot s_dot | A0 B0 A1 B1
constexpr unsigned F_DROP = 32u;    // silent drop (singular / non-finite / teleport), fp.py:826-833, :944-956

// ---- gated launch (host-pointer call) ------------------------------------------------------------------------------
// The sweep is launched before / while the obstacle tensor is uploaded in slices of gate_per queries; the upload streams
// set gate[slice] = gate_epoch behind each slice, and a CTA waits for the slice of its own query.
#ifndef FOT_GATE_SLEEP_NS
#define FOT_GATE_SLEEP_NS 1000
#endif
constexpr int kGateSlices = 64;
constexpr long long kGateTimeoutNs = 4000000000ll;   // a gated CTA gives up after 4 s (the host reports the error)

// Thread 0 waits until query q's slice has been uploaded; returns to every thread whether the CTA gave up (then
// gate[kGateSlices] is set for the host).  Geom: ItemGeom or PairGeom.
template <class Geom>
__device__ __forceinline__ bool gate_wait(const Geom& G, int q, int& s_abort) {
  if (threadIdx.x == 0) {
    const unsigned* flag = G.gate + (G.gate_q0 + q) / G.gate_per;
    int abort_ = 0;
    long long t0 = 0;
    for (unsigned spins = 0;; ++spins) {
      unsigned seen;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(flag) : "memory");
      if (seen == G.gate_epoch) break;
      __nanosleep(spins < 64 ? 100 : FOT_GATE_SLEEP_NS);
      long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      if (now - t0 > kGateTimeoutNs) { abort_ = 1; G.gate[kGateSlices] = 1u; break; }
    }
    asm volatile("fence.proxy.async.global;" ::: "memory");      // the bulk copy that follows reads what the upload wrote
    s_abort = abort_;
  }
  __syncthreads();
  return s_abort;
}

// Boxes of the predicted trajectories of a staged obstacle block (what fot_prepass does for a resident tensor): one
// warp per trajectory, fp32 rounded outward, NaN trajectory -> NaN box.
__device__ __forceinline__ void box_staged(const double2* dynst, float4* sbox, int SP, int T_obs, int warp, int n_warps, int lane) {
  for (int j = warp; j < SP; j += n_warps) {
    const double2* src = dynst + (size_t)j * T_obs;
    double xlo = INFINITY, xhi = -INFINITY, ylo = INFINITY, yhi = -INFINITY;
    bool bad = false;
    for (int k = lane; k < T_obs; k += 32) {
      const double2 o = src[k];
      bad |= (o.x != o.x) || (o.y != o.y);
      xlo = fmin(xlo, o.x); xhi = fmax(xhi, o.x); ylo = fmin(ylo, o.y); yhi = fmax(yhi, o.y);
    }
    for (int off = 16; off > 0; off >>= 1) {
      xlo = fmin(xlo, __shfl_xor_sync(0xffffffffu, xlo, off)); xhi = fmax(xhi, __shfl_xor_sync(0xffffffffu, xhi, off));
      ylo = fmin(ylo, __shfl_xor_sync(0xffffffffu, ylo, off)); yhi = fmax(yhi, __shfl_xor_sync(0xffffffffu, yhi, off));
    }
    bad = __any_sync(0xffffffffu, bad);
    if (lane == 0) {
      const float nanf_ = __int_as_float(0x7fc00000);
      sbox[j] = bad ? make_float4(nanf_, nanf_, nanf_, nanf_)
                    : make_float4(__double2float_rd(xlo), __double2float_ru(xhi), __double2float_rd(ylo), __double2float_ru(yhi));
    }
  }
}

// ---- the reference point ------------------------------------------------------------------------------------------
struct RefFast {
  double rx, ry, cth, sth, rk, rdk;
};
// Reference point at arc length s (cs.py:47-166, :215-288) with heading as a unit vector:
// cos(atan2(y', x')) = x'/|r'| (cc.py:128-129 takes cos/sin of the yaw).  NaN outside the knots.
// tab(k, i): entry i of table k (0 knots | 1-4 x: a b c d | 5-8 y: a b c d).
template <class Tab>
__device__ __forceinline__ RefFast spline_ref_tab(const Tab& tab, int nx, double s) {
  RefFast o;
  if (!(s >= tab(0, 0) && s <= tab(0, nx - 1))) {       // cs.py:62
    o.rx = o.ry = o.cth = o.sth = o.rk = o.rdk = qnan();
    return o;
  }
  int lo = 0, hi = nx;                                   // searchsorted(side='right') (cs.py:162)
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (tab(0, mid) <= s) lo = mid + 1; else hi = mid;
  }
  int seg = lo - 1;
  seg = seg < 0 ? 0 : (seg > nx - 2 ? nx - 2 : seg);     // cs.py:165
  const double dx = s - tab(0, seg);
  const double dx2 = dx * dx, dx3 = dx2 * dx;
  const double xa = tab(1, seg), xb = tab(2, seg), xc = tab(3, seg), xd = tab(4, seg);
  const double ya = tab(5, seg), yb = tab(6, seg), yc = tab(7, seg), yd = tab(8, seg);
  o.rx = xa + xb * dx + xc * dx2 + xd * dx3;             // cs.py:73-74
  o.ry = ya + yb * dx + yc * dx2 + yd * dx3;
  const double x1 = xb + 2.0 * xc * dx + 3.0 * xd * dx2; // cs.py:100
  const double y1 = yb + 2.0 * yc * dx + 3.0 * yd * dx2;
  const double x2 = 2.0 * xc + 6.0 * xd * dx;            // cs.py:125
  const double y2 = 2.0 * yc + 6.0 * yd * dx;
  const double x3 = 6.0 * xd, y3 = 6.0 * yd;             // cs.py:149
  const double D = x1 * x1 + y1 * y1;
  const double rD = rsqrt_nr(D);
  o.cth = x1 * rD;
  o.sth = y1 * rD;
  const double iD15 = rD * rD * rD;                      // D ** -1.5
  o.rk = (y2 * x1 - x2 * y1) * iD15;                     // cs.py:246
  const double a = x1 * y2 - y1 * x2;
  const double b = x1 * y3 - y1 * x3;
  const double c = x1 * x2 + y1 * y2;
  o.rdk = b * iD15 - 3.0 * a * c * (iD15 * rD * rD);     // cs.py:273
  return o;
}

// flag |= bit when a > b / when |a| > b: one DSETP and one predicated LOP3 (the compiler's own
// `cond ? bit : 0` idiom costs a SEL and a LOP3 per flag)
__device__ __forceinline__ void flag_gt(unsigned& f, double a, double b, unsigned bit) {
  asm("{\n .reg .pred p;\n setp.gt.f64 p, %1, %2;\n @p or.b32 %0, %0, %3;\n}" : "+r"(f) : "d"(a), "d"(b), "r"(bit));
}
__device__ __forceinline__ void flag_abs_gt(unsigned& f, double a, double b, unsigned bit) {
  asm("{\n .reg .pred p;\n .reg .f64 t;\n abs.f64 t, %1;\n setp.gt.f64 p, t, %2;\n @p or.b32 %0, %0, %3;\n}" : "+r"(f) : "d"(a), "d"(b), "r"(bit));
}

}  // namespace fot
