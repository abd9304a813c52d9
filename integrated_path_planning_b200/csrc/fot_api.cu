// fot_api.cu -- C ABI (include/fot.h) over the sweep kernels.  Host side only: argument
// checks, device tables, scratch, launches.  There is no CPU fallback anywhere in this file:
// without a CUDA device every entry point that computes returns FOT_ERR_NO_DEVICE.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <chrono>
#include <vector>
#include <mutex>
#include <set>
#include <initializer_list>

#include "fot_kernels.cuh"
#include "fot_sweep_items.cuh"
#include "fot_sweep_pairs.cuh"
#include "fot_predict.cuh"
#include "fot_frenet.cuh"
#include "fot_rank.cuh"
#include "fot_weights.cuh"
#include "fot_assess.cuh"
#include "fot_assess_cand.cuh"

using namespace fot;

namespace {

thread_local std::string g_err;

int fail(int code, const char* what, cudaError_t e = cudaSuccess) {
  char buf[512];
  if (e != cudaSuccess)
    snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
  else
    snprintf(buf, sizeof buf, "%s", what);
  g_err = buf;
  return code;
}

#define CK(call)                                                        \
  do {                                                                  \
    cudaError_t e__ = (call);                                           \
    if (e__ != cudaSuccess) return fail(FOT_ERR_CUDA, #call, e__);      \
  } while (0)

size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

// Growable device / pinned-host buffer.
struct Buf {
  void* p = nullptr;
  size_t cap = 0;
  bool host = false;
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    release();
    size_t want = n + n / 4 + 256;
    cudaError_t e = host ? cudaMallocHost(&p, want) : cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want; else p = nullptr;
    return e;
  }
  void release() {
    if (p) { if (host) cudaFreeHost(p); else cudaFree(p); }
    p = nullptr; cap = 0;
  }
};

// Tuning / test knobs (FOT_* environment variables).  They are resolved ONCE, when the handle is created -- no entry
// point reads the environment on the planning path -- and again only on an explicit fot_reload_options() (the tests
// and tuning scripts switch variants on a live handle that way).  Defaults are the product behaviour.
struct Options {
  int bpc = 0;                 // FOT_BPC            blocks per CTA (0: rule of item_geometry)
  int qcap = 1024;             // FOT_QCAP           collision queue entries (tests force the queue-full path)
  int fused_box = 0;           // FOT_FUSED_BOX      1: trajectory boxes in the sweep even for a resident tensor
  int stage_dyn = 1;           // FOT_STAGE_DYN      0: never stage the obstacle block in shared memory
  int sweep = 0;               // FOT_SWEEP          0 auto (fot_sweep_pairs, else fot_sweep_items), 1 "items", 4 "pairs" (fot_sweep_pairs:
                               //                    one longitudinal profile per warp, no block barriers; fail if unsupported)
  int pair_cpq = 0;            // FOT_PAIR_CPQ       CTAs per query of fot_sweep_pairs (0: rule of pair_geometry)
  int pair_simple = 1;         // FOT_PAIR_SIMPLE    0: always the instantiation of fot_sweep_pairs with every mode compiled in (tests)
  int pair_feat = 0;           // FOT_PAIR_FEAT      mode bits (PAIR_*) added to what the batch needs (tests, tuning)
  int host_chunks = 0;         // FOT_HOST_CHUNKS    equal chunks of the host-pointer call (0: rule)
  int gated = 1;               // FOT_GATED          0: chunked launches instead of gated ones
  int gate_uploads = 16;       // FOT_GATE_UPLOADS   upload slices of a gated call
  int gate_memcpy = 0;         // FOT_GATE_MEMCPY    1: flags by 4-byte copies instead of stream writes
  int debug_timing = 0;        // FOT_DEBUG_TIMING   1: print the timeline of every host-pointer call
  void resolve() {
    *this = Options{};
    auto geti = [](const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; };
    bpc = geti("FOT_BPC", 0);
    qcap = std::max(1, std::min(1 << 15, geti("FOT_QCAP", 1024)));
    fused_box = geti("FOT_FUSED_BOX", 0) != 0;
    stage_dyn = geti("FOT_STAGE_DYN", 1) != 0;
    if (const char* e = getenv("FOT_SWEEP")) sweep = !strcmp(e, "items") ? 1 : !strcmp(e, "pairs") ? 4 : 0;
    pair_cpq = geti("FOT_PAIR_CPQ", 0);
    pair_simple = geti("FOT_PAIR_SIMPLE", 1) != 0;
    pair_feat = geti("FOT_PAIR_FEAT", 0) & 31;
    host_chunks = geti("FOT_HOST_CHUNKS", 0);
    gated = geti("FOT_GATED", 1) != 0;
    gate_uploads = geti("FOT_GATE_UPLOADS", 16);
    gate_memcpy = getenv("FOT_GATE_MEMCPY") != nullptr;
    debug_timing = getenv("FOT_DEBUG_TIMING") != nullptr;
  }
};

std::mutex g_live_mu;
std::set<fot_handle*> g_live;     // handles alive in this process (fot_reload_options(NULL) walks them)

}  // namespace

// The instantiations of fot_sweep_pairs that exist (mode sets, PAIR_*), smallest first: the campaign shape, + static
// obstacles, + per-candidate outputs, + both, the unstaged obstacle block (large sample sets), the violation budget
// (chance-constrained planning), static obstacles + footprint (the corridor scenarios), everything; then the routed
// counterparts (PAIR_ROUTES, per-query reference paths) of the campaign shape, + static obstacles, + per-candidate outputs
// (top_k, cost weights) and everything.
#define FOT_PAIR_INSTANCES(X) X(0) X(PAIR_STATIC) X(PAIR_OUTPUTS) X(PAIR_STATIC | PAIR_OUTPUTS) X(PAIR_LOOSE) X(PAIR_BUDGET) \
  X(PAIR_STATIC | PAIR_FOOTPRINT) X(PAIR_ALL) X(PAIR_ROUTES) X(PAIR_ROUTES | PAIR_STATIC) X(PAIR_ROUTES | PAIR_OUTPUTS)     \
  X(PAIR_ROUTES | PAIR_ALL)
#define FOT_PAIR_LIST(f) (f),
static const int kPairInstances[] = {FOT_PAIR_INSTANCES(FOT_PAIR_LIST)};
static const int kPairInstanceCount = (int)(sizeof(kPairInstances) / sizeof(kPairInstances[0]));
typedef void (*PairKernel)(const Plan, const Batch, const Out, const PairGeom);
static PairKernel pair_kernel(bool fused, int feat) {
  switch (feat) {
#define FOT_PAIR_CASE(f) case (f): return fused ? fot_sweep_pairs<true, (f)> : fot_sweep_pairs<false, (f)>;
    FOT_PAIR_INSTANCES(FOT_PAIR_CASE)
    default:
      if (feat & PAIR_ROUTES) return fused ? fot_sweep_pairs<true, PAIR_ROUTES | PAIR_ALL> : fot_sweep_pairs<false, PAIR_ROUTES | PAIR_ALL>;
      return fused ? fot_sweep_pairs<true, PAIR_ALL> : fot_sweep_pairs<false, PAIR_ALL>;
  }
}

struct fot_handle {
  Options opt;
  int device = 0;
  Plan plan{};
  void* tables_dev = nullptr;
  cudaStream_t stream = nullptr, stream2 = nullptr, copy_stream = nullptr, d2h_stream = nullptr;
  static constexpr int kMaxChunks = 16;
  cudaEvent_t ev_copy[kMaxChunks] = {}, ev_done[kMaxChunks] = {};
  cudaEvent_t ev_join = nullptr, ev_blob = nullptr;
  cudaStream_t pstream[4] = {};      // gated launches: one stream per range of queries, earlier ranges at higher priority
  Buf gate_d, gate_h;                // gated launches: device progress / error words, pinned source words
  uint32_t gate_epoch = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool timed = false;
  static constexpr int kRing = 256;
  std::vector<cudaEvent_t> ring;     // kRing x 4 events: start, after prepass, after sweep, after winner
  long long n_launch = 0;
  int smem_optin = 0;
  int sms = 148;                     // SM count of the device (block-per-CTA grouping, host chunk sizes)
  Buf part_cost, part_idx, dyn_box, cost_tab;   // device scratch
  Buf w_pieces;                      // cost pieces of fot_select_weighted / fot_cost_terms (fot_weights.cuh)
  Buf ca_nan;                        // NaN bits of the pedestrian trajectories of fot_assess_candidates (fot_assess_cand.cuh)
  int last_pair_feat = -1;           // mode set (PAIR_*) of the fot_sweep_pairs instantiation of the last launch
  int last_sweep_kind = 0;           // 4: fot_sweep_pairs, 1: fot_sweep_items
  fot_result_t mirror{};             // fot_set_result_mirror: second destination of the winner block (all null: none)
  unsigned* mirror_flag = nullptr;   // word published behind each mirrored launch (fot_set_result_mirror), or null
  unsigned mirror_seq = 0;
  const double* last_winner_d = nullptr;   // full winner series of the last host-result call (device, in out_d)
  int last_winner_nq = 0;
  // routes (fot_add_route): host copies of the device tables of Routes, route 0 = the path of fot_create
  std::vector<double> rt_tab;        // every route's nine tables, nx doubles each
  std::vector<int32_t> rt_nx{0};     // [0] number of routes, [1 + r] knots of route r
  std::vector<int32_t> rt_off;       // [r] offset of route r in rt_tab
  int max_nx = 0;                    // most knots of any route: kernel choice and shared memory of a routed launch
  void* routes_dev = nullptr;        // rt_tab | rt_nx | rt_off on the device
  const int32_t* route_ids = nullptr;   // fot_set_routes: per-query route ids (device), null = no binding
  Buf stage_h, stage_d, out_d, dyn_d, stat_d;   // host-API staging
  fot_handle() { stage_h.host = true; gate_h.host = true; }
};

extern "C" int fot_abi_version(void) { return FOT_ABI_VERSION; }
extern "C" int fot_abi_minor(void) { return FOT_ABI_MINOR; }
extern "C" const char* fot_last_error(void) { return g_err.c_str(); }

extern "C" int fot_create(const fot_config_t* cfg, const fot_tables_t* tb, int device, fot_handle_t** out) {
  if (!cfg || !tb || !out) return fail(FOT_ERR_ARG, "fot_create: null argument");
  *out = nullptr;
  if (cfg->n_T < 1 || cfg->n_d < 1 || cfg->n_B < 0 || cfg->nx < 2 || cfg->n_total < 1 ||
      cfg->n_circles < 0 || cfg->n_circles > FOT_MAX_CIRCLES || !(cfg->dt > 0.0))
    return fail(FOT_ERR_ARG, "fot_create: bad grid sizes");
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0)
    return fail(FOT_ERR_NO_DEVICE, "fot_create: no CUDA device (this library has no CPU path)");
  if (device < 0 || device >= n_dev) return fail(FOT_ERR_ARG, "fot_create: bad device ordinal");
  CK(cudaSetDevice(device));

  fot_handle* h = new fot_handle();
  // any failure below releases everything created so far (streams, events, tables) through fot_destroy
  struct Guard { fot_handle* h; ~Guard() { if (h) fot_destroy(h); } } guard{h};
  h->opt.resolve();
  h->device = device;
  h->plan.cfg = *cfg;
  const int nT = cfg->n_T, nB = cfg->n_B, nd = cfg->n_d, nx = cfg->nx;
  int n_t_max = nB > 0 ? cfg->n_total : 0;
  for (int j = 0; j < nT; ++j) {
    if (tb->n_steps[j] < 1) return fail(FOT_ERR_ARG, "fot_create: horizon shorter than 2 samples");
    n_t_max = std::max(n_t_max, tb->n_steps[j] + 1);
  }
  for (int j = 0; j < nB; ++j)
    if (tb->n_steps_b[j] + 1 > cfg->n_total) return fail(FOT_ERR_ARG, "fot_create: brake horizon longer than max_t");
  h->plan.n_t_max = n_t_max;
  h->plan.d_sorted = 1;
  h->plan.d_min = h->plan.d_max = tb->d_grid[0];
  for (int i = 0; i < nd; ++i) {
    if (i > 0 && !(tb->d_grid[i] >= tb->d_grid[i - 1])) h->plan.d_sorted = 0;
    h->plan.d_min = std::min(h->plan.d_min, tb->d_grid[i]);
    h->plan.d_max = std::max(h->plan.d_max, tb->d_grid[i]);
  }

  // one device blob: doubles first, then the int tables
  std::vector<double> dbl;
  auto push = [&](const double* p, size_t n) { size_t o = dbl.size(); dbl.insert(dbl.end(), p, p + n); return o; };
  const size_t oT = push(tb->T, nT), oI4 = push(tb->inv4, 4 * (size_t)nT), oI5 = push(tb->inv5, 9 * (size_t)nT);
  const size_t oTb = nB ? push(tb->Tb, nB) : 0, oI4b = nB ? push(tb->inv4b, 4 * (size_t)nB) : 0,
               oI5b = nB ? push(tb->inv5b, 9 * (size_t)nB) : 0;
  const size_t oD = push(tb->d_grid, nd), oK = push(tb->knots, nx);
  const size_t oxa = push(tb->xa, nx), oxb = push(tb->xb, nx - 1), oxc = push(tb->xc, nx), oxd = push(tb->xd, nx - 1);
  const size_t oya = push(tb->ya, nx), oyb = push(tb->yb, nx - 1), oyc = push(tb->yc, nx), oyd = push(tb->yd, nx - 1);
  std::vector<int32_t> ints(tb->n_steps, tb->n_steps + nT);
  if (nB) ints.insert(ints.end(), tb->n_steps_b, tb->n_steps_b + nB);
  const size_t dbytes = dbl.size() * sizeof(double), ibytes = ints.size() * sizeof(int32_t);
  cudaError_t e = cudaMalloc(&h->tables_dev, dbytes + ibytes);
  if (e != cudaSuccess) { h->tables_dev = nullptr; return fail(FOT_ERR_CUDA, "cudaMalloc(tables)", e); }
  e = cudaMemcpy(h->tables_dev, dbl.data(), dbytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy((char*)h->tables_dev + dbytes, ints.data(), ibytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return fail(FOT_ERR_CUDA, "cudaMemcpy(tables)", e);
  const double* D = (const double*)h->tables_dev;
  const int32_t* I = (const int32_t*)((char*)h->tables_dev + dbytes);
  Plan& P = h->plan;
  P.T = D + oT; P.inv4 = D + oI4; P.inv5 = D + oI5;
  P.Tb = D + oTb; P.inv4b = D + oI4b; P.inv5b = D + oI5b;
  P.d_grid = D + oD; P.knots = D + oK;
  P.xa = D + oxa; P.xb = D + oxb; P.xc = D + oxc; P.xd = D + oxd;
  P.ya = D + oya; P.yb = D + oyb; P.yc = D + oyc; P.yd = D + oyd;
  P.n_steps = I; P.n_steps_b = I + nT;
  {
    const fot_route_t r0{nx, tb->knots, tb->xa, tb->xb, tb->xc, tb->xd, tb->ya, tb->yb, tb->yc, tb->yd};
    int32_t id = 0;
    const int rc = fot_add_route(h, &r0, &id);
    if (rc != FOT_OK) return rc;
  }

  CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_blob, cudaEventDisableTiming));
  {
    int least = 0, greatest = 0;
    CK(cudaDeviceGetStreamPriorityRange(&least, &greatest));     // numerically lower = higher priority
    for (int i = 0; i < 4; ++i)
      CK(cudaStreamCreateWithPriority(&h->pstream[i], cudaStreamNonBlocking, std::min(least, greatest + i)));
  }
  CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking));
  for (auto& ev : h->ev_copy) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  for (auto& ev : h->ev_done) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  CK(cudaEventCreate(&h->ev0));
  CK(cudaEventCreate(&h->ev1));
  h->ring.resize((size_t)fot_handle::kRing * 4);
  for (auto& ev : h->ring) CK(cudaEventCreate(&ev));
  CK(cudaDeviceGetAttribute(&h->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  CK(cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, device));
  h->smem_optin -= 2048;   // leave room for the kernels' static shared memory
  CK(cudaFuncSetAttribute(fot_sweep_items<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem_optin));
  CK(cudaFuncSetAttribute(fot_sweep_items<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem_optin));
  CK(cudaFuncSetAttribute(fot_sweep_items<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem_optin));
  CK(cudaFuncSetAttribute(fot_sweep_items<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem_optin));
  for (int i = 0; i < kPairInstanceCount; ++i)
    for (int f = 0; f < 2; ++f)
      CK(cudaFuncSetAttribute(pair_kernel(f != 0, kPairInstances[i]), cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem_optin));
  { std::lock_guard<std::mutex> lk(g_live_mu); g_live.insert(h); }
  guard.h = nullptr;
  *out = h;
  return FOT_OK;
}

extern "C" int fot_reload_options(fot_handle_t* h) {
  std::lock_guard<std::mutex> lk(g_live_mu);
  if (h) { if (!g_live.count(h)) return fail(FOT_ERR_ARG, "fot_reload_options: unknown handle"); h->opt.resolve(); return FOT_OK; }
  for (fot_handle* x : g_live) x->opt.resolve();
  return FOT_OK;
}

extern "C" int fot_destroy(fot_handle_t* h) {
  if (!h) return FOT_OK;
  { std::lock_guard<std::mutex> lk(g_live_mu); g_live.erase(h); }
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();          // every stream of the handle (compute, priority, copy) is idle before its buffers go
  for (Buf* b : {&h->gate_d, &h->gate_h, &h->part_cost, &h->part_idx, &h->dyn_box, &h->cost_tab, &h->w_pieces, &h->ca_nan, &h->stage_h,
                 &h->stage_d, &h->out_d, &h->dyn_d, &h->stat_d})
    b->release();
  if (h->tables_dev) cudaFree(h->tables_dev);
  if (h->routes_dev) cudaFree(h->routes_dev);
  for (auto ev : h->ring) if (ev) cudaEventDestroy(ev);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  for (auto ev : h->ev_copy) if (ev) cudaEventDestroy(ev);
  for (auto ev : h->ev_done) if (ev) cudaEventDestroy(ev);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->ev_blob) cudaEventDestroy(h->ev_blob);
  for (auto ps : h->pstream) if (ps) cudaStreamDestroy(ps);
  if (h->stream2) cudaStreamDestroy(h->stream2);
  if (h->d2h_stream) cudaStreamDestroy(h->d2h_stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return FOT_OK;
}

extern "C" int fot_n_t_max(const fot_handle_t* h) { return h ? h->plan.n_t_max : FOT_ERR_ARG; }

extern "C" int fot_candidate_count(const fot_handle_t* h, int n_v, int has_brake) {
  if (!h || n_v < 0) return FOT_ERR_ARG;
  return h->plan.cfg.n_T * n_v * h->plan.cfg.n_d + (has_brake ? h->plan.cfg.n_B : 0);
}

// Knots of the path(s) a launch sweeps: with a route binding the longest route's (fot_set_routes), else the handle's path.
static int sweep_nx(const fot_handle* h) { return h->route_ids ? h->max_nx : h->plan.cfg.nx; }

// The Routes of a launch whose first query is query q_off of the bound route array (all null without a binding).
static Routes routes_of(const fot_handle* h, size_t q_off) {
  Routes R{};
  if (!h->route_ids) return R;
  const size_t n_routes = h->rt_off.size();
  R.id = h->route_ids + q_off;
  R.tab = (const double*)h->routes_dev;
  R.nx = (const int32_t*)(R.tab + h->rt_tab.size());
  R.off = R.nx + 1 + n_routes;
  return R;
}

// Geometry of the sample-major kernel (fot_sweep_items).  Returns false, with the limit that was exceeded in
// fot_last_error, when the batch's shape is outside what that kernel covers: then no sweep kernel takes it.
static bool item_geometry(const fot_handle* h, const fot_batch_t* b, ItemGeom* g, size_t* smem_bytes,
                          bool want_fused_box = false) {
  const int NT = h->plan.n_t_max, nd = h->plan.cfg.n_d, nB = h->plan.cfg.n_B, nx = sweep_nx(h);
  const bool has_dyn = b->dyn_mode != FOT_DYN_NONE;
  const long long SPl = has_dyn ? (long long)b->S * b->P : 0;
  char why[160];
  if (NT > kItemThreads)
    snprintf(why, sizeof why, "time grid of %d samples: the sweep takes at most %d", NT, kItemThreads);
  else if (nd > 8192)
    snprintf(why, sizeof why, "lateral grid of %d targets: the sweep takes at most 8192", nd);
  else if (SPl > 32768)
    snprintf(why, sizeof why, "%lld obstacle trajectories (S*P): the sweep takes at most 32768", SPl);
  else if (b->n_static > 32768)
    snprintf(why, sizeof why, "%d static obstacle points: the sweep takes at most 32768", b->n_static);
  else
    why[0] = 0;
  if (why[0]) { fail(FOT_ERR_TOO_LARGE, why); return false; }
  const int SP = (int)SPl;
  const int ppc_max = kItemThreads / NT;
  ItemGeom G{};
  G.chunks = (b->n_v_max + ppc_max - 1) / ppc_max;
  G.ppc = (b->n_v_max + G.chunks - 1) / G.chunks;
  G.grid_blocks = h->plan.cfg.n_T * G.chunks;
  G.ppb = nB > 0 ? std::min(nB, ppc_max) : 0;
  G.brake_blocks = nB > 0 ? (nB + G.ppb - 1) / G.ppb : 0;
  G.blocks_per_query = G.grid_blocks + G.brake_blocks;
  // blocks per CTA: a whole query per CTA once the batch alone fills the GPU several times over,
  // one block per CTA for single plan() calls
  {
    const int sms = h->sms;
    const long long total = (long long)b->n_q * G.blocks_per_query;
    long long bpc = total / ((long long)sms * 2 * 4);
    bpc = std::max<long long>(1, std::min<long long>(bpc, G.blocks_per_query));
    if (h->opt.bpc > 0) bpc = std::max(1, std::min(h->opt.bpc, (int)G.blocks_per_query));
    G.ctas_per_query = (int)((G.blocks_per_query + bpc - 1) / bpc);
    G.bpc = (G.blocks_per_query + G.ctas_per_query - 1) / G.ctas_per_query;
  }
  G.pcap = std::max(G.ppc, std::max(G.ppb, 1));
  G.threads = (G.pcap * NT + 31) / 32 * 32;
  G.ct_lcap = std::max(nd, std::max(G.ppb, 1));
  G.nw4 = (nd + 3) / 4;
  G.nwc = (nd + 31) / 32;
  const int max_viol = b->dyn_mode == FOT_DYN_DISTRIBUTION ? (int)std::floor(h->plan.cfg.chance_epsilon * (double)b->S) : 0;
  G.vwords = max_viol > 0 ? (b->S + 31) / 32 : 0;
  G.lcap = std::max(1, SP + b->n_static);
  G.ochunk = G.lcap <= 256 ? G.lcap : 128;
  G.qcap = h->opt.qcap;                   // (the tests shrink it to force the queue-full path)
  G.spline_smem = nx <= 128 ? 1 : 0;
  const size_t dyn_bytes = (size_t)SP * b->T_obs * 16;
  // option fused_box (tests, tuning): trajectory boxes in the sweep even for a resident tensor
  const bool fuse = want_fused_box || h->opt.fused_box;
  auto layout = [&](bool stage) {
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 15) / 16 * 16; return (int32_t)o; };
    G.o_row = take((size_t)G.pcap * NT * kRowW * 8);
    G.o_sdl = take((size_t)G.pcap * 8);
    G.o_ct = take((size_t)(G.pcap + 2 * G.ct_lcap) * 8);
    G.o_dgrid = take((size_t)nd * 8);
    G.o_vlast = take((size_t)G.pcap * nd * 8);
    G.o_spl = take(G.spline_smem ? (size_t)9 * nx * 8 : 0);
    G.o_dyn = take(stage ? dyn_bytes : 0);
    G.o_box = take(stage && fuse ? (size_t)SP * 16 : 0);
    G.o_fn = take((size_t)G.pcap * 4);
    G.o_flags = take((size_t)G.pcap * G.nw4 * 4);
    G.o_hit = take((size_t)G.pcap * G.nwc * 4);
    G.o_viol = take((size_t)G.pcap * nd * G.vwords * 4);
    G.n_zero = (int32_t)((off - (size_t)G.o_flags) / 4);
    G.o_queue = take((size_t)G.qcap * 4);
    G.o_list = take((size_t)G.lcap * 4);
    G.o_clean = take((size_t)G.pcap * G.nwc * 4);
    G.o_slow = take((size_t)G.threads * 2);
    G.stage_dyn = stage ? 1 : 0;
    G.fused_box = stage && fuse ? 1 : 0;
    return off;
  };
  // stage the query's obstacle block in shared memory when two blocks per SM still fit
  bool stage = has_dyn && dyn_bytes > 0 && dyn_bytes <= 64 * 1024 && ((uintptr_t)b->dyn & 15) == 0;
  stage = stage && h->opt.stage_dyn;
  size_t bytes = layout(stage);
  if (stage && bytes > 110 * 1024) { stage = false; bytes = layout(false); }
  if (bytes > (size_t)h->smem_optin) {
    snprintf(why, sizeof why, "sweep tables of %zu bytes: a block has %d bytes of shared memory", bytes, h->smem_optin);
    fail(FOT_ERR_TOO_LARGE, why);
    return false;
  }
  *g = G;
  *smem_bytes = bytes;
  return true;
}

// Geometry of the pair-per-warp kernel (fot_sweep_pairs): one CTA per query (several for small batches), every warp
// with a private slice of shared memory for the pair it is working on.  False when the shape is outside its range
// (time grids beyond kPairNT = 56 samples, lateral grids beyond 96 targets, tables that do not fit): fot_sweep_items then runs.
static bool pair_geometry(const fot_handle* h, const fot_batch_t* b, PairGeom* g, size_t* smem_bytes,
                          bool want_fused_box = false) {
  const int NT = h->plan.n_t_max, nd = h->plan.cfg.n_d, nB = h->plan.cfg.n_B, nx = sweep_nx(h);
  const bool has_dyn = b->dyn_mode != FOT_DYN_NONE;
  const long long SPl = has_dyn ? (long long)b->S * b->P : 0;
  if (NT > kPairNT || nd > kPairND || b->n_v_max > kPairNV || nx > kPairNX || h->plan.cfg.n_T > kPairNH || SPl > (1 << 20) || b->n_static > (1 << 20)) return false;
  if (SPl * std::max(1, b->T_obs) >= (1ll << 27)) return false;                            // list entries: element offsets
  const int SP = (int)SPl;
  PairGeom G{};
  G.nw4 = (nd + 3) / 4;
  G.nwc = (nd + 31) / 32;
  const int max_viol = b->dyn_mode == FOT_DYN_DISTRIBUTION ? (int)std::floor(h->plan.cfg.chance_epsilon * (double)b->S) : 0;
  G.vwords = max_viol > 0 ? (b->S + 31) / 32 : 0;
  G.viol_bytes = (nd * G.vwords * 4 + 15) / 16 * 16;
  const size_t dyn_bytes = (size_t)SP * b->T_obs * 16;
  const bool fuse = want_fused_box || h->opt.fused_box;
  auto layout = [&](bool stage) {
    size_t off = sizeof(PairShared);
    auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 15) / 16 * 16; return (int32_t)o; };
    const bool box = has_dyn && ((stage && fuse) || (size_t)SP * 16 <= 8 * 1024);
    G.o_dyn = take(stage ? dyn_bytes : 0);
    G.o_box = take(box ? (size_t)SP * 16 : 0);
    G.o_viol = take((size_t)kPairWarps * G.viol_bytes);
    G.stage_dyn = stage ? 1 : 0;
    G.fused_box = stage && fuse ? 1 : 0;
    G.box_smem = box ? 1 : 0;
    return off;
  };
  // stage the query's obstacle block in shared memory when two CTAs per SM still fit
  bool stage = has_dyn && dyn_bytes > 0 && dyn_bytes <= 64 * 1024 && ((uintptr_t)b->dyn & 15) == 0;
  stage = stage && h->opt.stage_dyn;
  size_t bytes = layout(stage);
  if (stage && bytes > 113 * 1024 - 512) { stage = false; bytes = layout(false); }
  if (bytes > (size_t)h->smem_optin) return false;
  // CTAs per query: one once the batch alone fills the GPU several times over; for small batches the pairs of a
  // query are dealt to several CTAs (about one pair per warp for a single plan() call)
  {
    const int n_units = h->plan.cfg.n_T * b->n_v_max + nB;
    long long cpq = ((long long)h->sms * 2 * 4 + b->n_q - 1) / b->n_q;
    cpq = std::max<long long>(1, std::min<long long>(cpq, (n_units + kPairWarps - 1) / kPairWarps));
    if (h->opt.pair_cpq > 0) cpq = std::max(1, std::min(h->opt.pair_cpq, n_units));
    G.ctas_per_query = (int)cpq;
  }
  *g = G;
  *smem_bytes = bytes;
  return true;
}

// The sweep kernel of a launch, with its geometry and dynamic shared memory.  kind takes the values of
// fot_last_sweep_kind (and of Options::sweep).
enum SweepKind { kItems = 1, kPairs = 4 };
struct Sweep {
  int kind = 0;
  ItemGeom ig{};      // fot_sweep_items; for fot_sweep_pairs the scratch layout it shares with it
  PairGeom pg{};      // fot_sweep_pairs
  size_t smem = 0;
};

// Kernel choice: the pair-per-warp fot_sweep_pairs wherever its shape limits allow, else the sample-major
// fot_sweep_items.  FOT_SWEEP=pairs / items insists on one of them (the tests cross-check the two).  A shape beyond
// fot_sweep_items is FOT_ERR_TOO_LARGE: fot_sweep_pairs needs its scratch layout.  A gated launch needs a sweep with a
// staged obstacle block: the gate of fot_sweep_items decides that, and fot_sweep_pairs runs gated only where it stages
// the block too.
static int select_sweep(const fot_handle* h, const fot_batch_t* b, bool gated, Sweep* s) {
  *s = Sweep{};
  size_t ismem = 0, psmem = 0;
  if (!item_geometry(h, b, &s->ig, &ismem, gated)) return FOT_ERR_TOO_LARGE;
  if (gated && !s->ig.fused_box) return fail(FOT_ERR_ARG, "gated launch needs a sample-major sweep with a staged obstacle block");
  const bool pairs = (h->opt.sweep == 0 || h->opt.sweep == kPairs) && pair_geometry(h, b, &s->pg, &psmem, gated) &&
                     (!gated || s->pg.fused_box);
  if (h->opt.sweep == kPairs && !pairs && !gated) return fail(FOT_ERR_ARG, "FOT_SWEEP=pairs: shape not supported by fot_sweep_pairs");
  if (pairs) {
    // same scratch (cost tables, trajectory boxes, one arg-min partial per CTA) as fot_sweep_items
    s->ig.blocks_per_query = h->plan.cfg.n_T * b->n_v_max + h->plan.cfg.n_B;      // upper bound of ctas_per_query (scratch stride)
    s->ig.ctas_per_query = s->pg.ctas_per_query; s->ig.threads = kPairThreads;
    s->ig.fused_box = s->pg.fused_box;
    s->kind = kPairs;
    s->smem = psmem;
  } else {
    s->kind = kItems;
    s->smem = ismem;
  }
  return FOT_OK;
}

static int check_batch(const fot_handle* h, const fot_batch_t* b, const fot_result_t* r) {
  if (!h || !b || !r) return fail(FOT_ERR_ARG, "null argument");
  if (b->n_q < 1 || b->n_v_max < 1) return fail(FOT_ERR_ARG, "n_q and n_v_max must be >= 1");
  if (!b->frenet || !b->target_speed || !b->limits || !b->stop_dist || !b->v_grid || !b->n_v)
    return fail(FOT_ERR_ARG, "null query array");
  if (b->n_static < 0 || (b->n_static > 0 && !b->static_obs)) return fail(FOT_ERR_ARG, "static obstacles missing");
  if (b->dyn_mode != FOT_DYN_NONE) {
    if (b->dyn_mode != FOT_DYN_SINGLE && b->dyn_mode != FOT_DYN_DISTRIBUTION) return fail(FOT_ERR_ARG, "bad dyn_mode");
    if (!b->dyn || b->S < 1 || b->P < 1 || b->T_obs < 1) return fail(FOT_ERR_ARG, "dynamic obstacle shape");
    if (b->dyn_mode == FOT_DYN_SINGLE && b->S != 1) return fail(FOT_ERR_ARG, "single-sample mode needs S == 1");
    if (b->dyn_mode == FOT_DYN_DISTRIBUTION && b->S > 64 &&
        std::floor(h->plan.cfg.chance_epsilon * (double)b->S) > 0.0)
      return fail(FOT_ERR_ARG, "chance_epsilon > 0 supports at most 64 samples");
  }
  if (!r->best_idx || !r->best_cost || !r->stats || !r->winner_len || !r->winner)
    return fail(FOT_ERR_ARG, "null result array");
  if ((r->cand_cat || r->cand_cost) && r->cand_stride < fot_candidate_count(h, b->n_v_max, 1))
    return fail(FOT_ERR_ARG, "cand_stride too small");
  if (r->winner_samples < 0) return fail(FOT_ERR_ARG, "winner_samples must be >= 0");
  return FOT_OK;
}

// q_off / q_total: this launch handles queries [q_off, q_off + b->n_q) of a batch of q_total whose chunks may be
// in flight on two streams at once, so every scratch buffer is sized for the batch and addressed by q_off.
// cuStreamWriteValue32 through the runtime's driver entry-point lookup (no link-time dependency on libcuda): a
// stream-ordered 4-byte write with a memory fence before it, far cheaper than a 4-byte cudaMemcpyAsync.
typedef int (*StreamWrite32)(cudaStream_t, unsigned long long, unsigned, unsigned);
static StreamWrite32 stream_write32() {
  static StreamWrite32 fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr{};
    if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &p, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (StreamWrite32)p;
  }();
  return fn;
}

struct Gate {
  unsigned* word = nullptr;      // device slice flags (nullptr: not gated)
  uint32_t epoch = 0;
  int per = 1;                   // queries per upload slice
};

static int launch_all(fot_handle* h, const fot_batch_t* b, const fot_result_t* r, cudaStream_t st, size_t q_off = 0,
                      size_t q_total = 0, Gate gate = Gate{}, bool record_span = true) {
  if (q_total == 0) q_total = (size_t)b->n_q;
  Sweep s;
  const int rc = select_sweep(h, b, gate.word != nullptr, &s);
  if (rc != FOT_OK) return rc;
  ItemGeom& ig = s.ig;
  PairGeom& pg = s.pg;
  if (gate.word) {
    ig.gate = gate.word; ig.gate_epoch = gate.epoch; ig.gate_per = gate.per; ig.gate_q0 = (int32_t)q_off;
    pg.gate = gate.word; pg.gate_epoch = gate.epoch; pg.gate_per = gate.per; pg.gate_q0 = (int32_t)q_off;
  }
  const bool has_dyn = b->dyn_mode != FOT_DYN_NONE;
  const size_t n_part = (size_t)b->n_q * ig.ctas_per_query;
  if (n_part > 0x7fffffffull) return fail(FOT_ERR_ARG, "batch too large for one launch");
  // partial winners: chunks of one batch may cut their queries into different numbers of CTAs; the stride that
  // addresses the scratch is the largest any chunk can use
  const size_t part_stride = (size_t)std::max(ig.blocks_per_query, ig.ctas_per_query);
  CK(h->part_cost.reserve(q_total * part_stride * sizeof(double)));
  CK(h->part_idx.reserve(q_total * part_stride * sizeof(int32_t)));
  const int SP = has_dyn ? b->S * b->P : 0;
  const bool need_box = has_dyn && !ig.fused_box;
  const size_t cost_stride = (size_t)h->plan.cfg.n_T * (b->n_v_max + 2 * h->plan.cfg.n_d) + 3 * (size_t)h->plan.cfg.n_B;
  if (need_box) CK(h->dyn_box.reserve(q_total * SP * sizeof(float4)));
  CK(h->cost_tab.reserve(q_total * cost_stride * sizeof(double)));
  float4* dyn_box = need_box ? (float4*)h->dyn_box.p + q_off * SP : nullptr;
  double* cost_tab = (double*)h->cost_tab.p + q_off * cost_stride;

  Batch B{};
  B.n_q = b->n_q; B.n_v_max = b->n_v_max;
  B.frenet = b->frenet; B.target = b->target_speed; B.limits = b->limits; B.stop_dist = b->stop_dist;
  B.v_grid = b->v_grid; B.n_v = b->n_v;
  B.n_static = b->n_static; B.static_per_query = b->static_per_query;
  B.S = has_dyn ? b->S : 0; B.P = has_dyn ? b->P : 0; B.T_obs = has_dyn ? b->T_obs : 0; B.dyn_mode = b->dyn_mode;
  B.dyn_raw = has_dyn ? b->dyn : nullptr;
  B.static_raw = b->n_static > 0 ? b->static_obs : nullptr;
  B.dyn_box = dyn_box;
  B.cost_tab = cost_tab;
  B.rt = routes_of(h, q_off);
  Out O{};
  O.best_idx = r->best_idx; O.best_cost = r->best_cost; O.stats = r->stats; O.winner_len = r->winner_len;
  O.winner = r->winner; O.cand_cat = r->cand_cat; O.cand_cost = r->cand_cost; O.cand_stride = r->cand_stride;
  O.part_cost = (double*)h->part_cost.p + q_off * part_stride; O.part_idx = (int32_t*)h->part_idx.p + q_off * part_stride;
  if (h->mirror.winner && q_off == 0 && q_total == (size_t)b->n_q) {     // whole-batch launches only (fot_plan_batch_device)
    O.m_best_idx = h->mirror.best_idx; O.m_best_cost = h->mirror.best_cost; O.m_stats = h->mirror.stats;
    O.m_winner_len = h->mirror.winner_len; O.m_winner = h->mirror.winner;
  }

  cudaEvent_t* ring = h->ring.data() + (size_t)(h->n_launch % fot_handle::kRing) * 4;
  if (record_span) CK(cudaEventRecord(h->ev0, st));
  {
    const size_t n_cat = r->cand_cat ? (size_t)b->n_q * r->cand_stride : 0;
    const size_t work = std::max<size_t>((size_t)b->n_q * FOT_N_STATS, n_cat);
    const int blocks = (int)std::min<size_t>(1024, (work + 255) / 256);
    fot_init_kernel<<<blocks, 256, 0, st>>>(r->stats, b->n_q * FOT_N_STATS, r->cand_cat, n_cat);
  }
  CK(cudaEventRecord(ring[0], st));
  {
    // cost tables (one thread per polynomial profile) and trajectory boxes (one warp per trajectory), one launch
    const long long n_prof = (long long)h->plan.cfg.n_T * (b->n_v_max + h->plan.cfg.n_d) + 2 * h->plan.cfg.n_B;
    const long long cblocks = ((long long)b->n_q * n_prof + 255) / 256;
    const long long n_traj = need_box ? (long long)b->n_q * SP : 0;
    const long long ablocks = ((n_traj + kBoxPerWarp - 1) / kBoxPerWarp * 32 + 255) / 256;
    if (cblocks + ablocks > 0x7fffffffll) return fail(FOT_ERR_ARG, "batch too large for one launch");
    fot_prepass<<<(unsigned)(cblocks + ablocks), 256, 0, st>>>(h->plan, B, cost_tab, (unsigned)cblocks,
                                                               (const double2*)b->dyn, dyn_box, n_traj, b->T_obs);
  }
  CK(cudaEventRecord(ring[1], st));
  if (s.kind == kPairs) {
    // the modes this batch needs; the smallest instantiated superset runs (everything else is compiled out of it)
    int need = 0;
    if (b->n_static > 0) need |= PAIR_STATIC;
    if (h->plan.cfg.n_circles > 0) need |= PAIR_FOOTPRINT;
    if (pg.vwords > 0) need |= PAIR_BUDGET;
    if (r->cand_cat || r->cand_cost) need |= PAIR_OUTPUTS;
    if (has_dyn && !(pg.stage_dyn && pg.box_smem)) need |= PAIR_LOOSE;
    if (!h->plan.d_sorted) need |= PAIR_LOOSE;
    need |= h->opt.pair_feat;
    if (!h->opt.pair_simple) need = PAIR_ALL;
    if (B.rt.id) need |= PAIR_ROUTES;
    int feat = PAIR_ALL | (need & PAIR_ROUTES);
    for (int i = 0; i < kPairInstanceCount; ++i)
      if ((kPairInstances[i] & need) == need) { feat = kPairInstances[i]; break; }
    pair_kernel(pg.fused_box != 0, feat)<<<(unsigned)n_part, kPairThreads, s.smem, st>>>(h->plan, B, O, pg);
    h->last_pair_feat = feat;
  } else {
    auto items = B.rt.id ? (ig.fused_box ? fot_sweep_items<true, true> : fot_sweep_items<false, true>)
                         : (ig.fused_box ? fot_sweep_items<true> : fot_sweep_items<false>);
    items<<<(unsigned)n_part, ig.threads, s.smem, st>>>(h->plan, B, O, ig);
  }
  h->last_sweep_kind = s.kind;
  CK(cudaEventRecord(ring[2], st));
  fot_winner<<<b->n_q, 128, (size_t)kTT * h->plan.n_t_max * sizeof(double), st>>>(h->plan, B, O, ig.ctas_per_query);
  if (O.m_winner && h->mirror_flag) fot_publish_kernel<<<1, 1, 0, st>>>(h->mirror_flag, ++h->mirror_seq);
  CK(cudaEventRecord(ring[3], st));
  if (record_span) CK(cudaEventRecord(h->ev1, st));
  h->n_launch++;
  CK(cudaGetLastError());
  h->timed = true;
  return FOT_OK;
}

extern "C" int fot_plan_batch_device(fot_handle_t* h, const fot_batch_t* b, const fot_result_t* r, void* stream) {
  int rc = check_batch(h, b, r);
  if (rc != FOT_OK) return rc;
  CK(cudaSetDevice(h->device));
  if (r->winner_samples != 0) return fail(FOT_ERR_ARG, "winner_samples applies to the host-result entry points only");
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  rc = launch_all(h, b, r, st);
  if (rc != FOT_OK) return rc;
  if (!stream) CK(cudaStreamSynchronize(st));
  return FOT_OK;
}

extern "C" int fot_rank_candidates(fot_handle_t* h, const fot_batch_t* b, const uint8_t* cand_cat, const double* cand_cost,
                                   int cand_stride, const fot_ranked_t* out, void* stream) {
  if (!h || !b || !out || !cand_cat || !cand_cost) return fail(FOT_ERR_ARG, "fot_rank_candidates: null argument");
  if (b->n_q < 1 || b->n_v_max < 1) return fail(FOT_ERR_ARG, "fot_rank_candidates: n_q and n_v_max must be >= 1");
  if (out->k < 1 || out->k > FOT_MAX_RANKED) return fail(FOT_ERR_ARG, "fot_rank_candidates: k must be in [1, FOT_MAX_RANKED]");
  if (!out->idx || !out->cost) return fail(FOT_ERR_ARG, "fot_rank_candidates: null idx or cost");
  if (out->series && !out->len) return fail(FOT_ERR_ARG, "fot_rank_candidates: series needs len");
  if (cand_stride < fot_candidate_count(h, b->n_v_max, 1)) return fail(FOT_ERR_ARG, "fot_rank_candidates: cand_stride too small");
  if (out->len && (!b->frenet || !b->v_grid || !b->n_v)) return fail(FOT_ERR_ARG, "fot_rank_candidates: null query array");
  if ((size_t)b->n_q * out->k > 0x7fffffffull) return fail(FOT_ERR_ARG, "fot_rank_candidates: batch too large for one launch");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  const Ranked R{out->k, out->idx, out->cost, out->len, out->series};
  fot_rank<<<b->n_q, kRankThreads, 0, st>>>(cand_cat, cand_cost, cand_stride, R);
  if (out->len) {
    Batch B{};
    B.n_q = b->n_q; B.n_v_max = b->n_v_max;
    B.frenet = b->frenet; B.v_grid = b->v_grid; B.n_v = b->n_v;
    B.rt = routes_of(h, 0);
    fot_rank_series<<<(unsigned)((size_t)b->n_q * out->k), 128, (size_t)kTT * h->plan.n_t_max * sizeof(double), st>>>(h->plan, B, R);
  }
  CK(cudaGetLastError());
  if (!stream) CK(cudaStreamSynchronize(st));
  return FOT_OK;
}

extern "C" int fot_assess_trajectories(fot_handle_t* h, const fot_batch_t* b, const fot_assessed_t* a, void* stream) {
  if (!h || !b || !a) return fail(FOT_ERR_ARG, "fot_assess_trajectories: null argument");
  if (b->n_q < 1) return fail(FOT_ERR_ARG, "fot_assess_trajectories: n_q must be >= 1");
  if (a->m < 1 || a->m > FOT_MAX_ASSESSED) return fail(FOT_ERR_ARG, "fot_assess_trajectories: m must be in [1, FOT_MAX_ASSESSED]");
  if (a->n_t < 1 || a->n_t > FOT_MAX_ASSESS_NT)
    return fail(FOT_ERR_ARG, "fot_assess_trajectories: n_t must be in [1, FOT_MAX_ASSESS_NT]");
  if (a->n_r < 1 || a->n_r > FOT_MAX_RADII) return fail(FOT_ERR_ARG, "fot_assess_trajectories: n_r must be in [1, FOT_MAX_RADII]");
  if (!a->series || !a->len) return fail(FOT_ERR_ARG, "fot_assess_trajectories: null series or len");
  if (!a->r2) return fail(FOT_ERR_ARG, "fot_assess_trajectories: null r2");
  if (!a->dyn_min || !a->dyn_at || !a->static_min || !a->static_at || !a->dyn_hits || !a->first_hit || !a->static_hit)
    return fail(FOT_ERR_ARG, "fot_assess_trajectories: null output array");
  if (b->n_static < 0 || b->S < 0 || b->P < 0 || b->T_obs < 0)
    return fail(FOT_ERR_ARG, "fot_assess_trajectories: negative obstacle shape");
  if (b->n_static > 0 && !b->static_obs) return fail(FOT_ERR_ARG, "fot_assess_trajectories: static obstacles missing");
  if (b->dyn_mode != FOT_DYN_NONE && b->dyn_mode != FOT_DYN_SINGLE && b->dyn_mode != FOT_DYN_DISTRIBUTION)
    return fail(FOT_ERR_ARG, "fot_assess_trajectories: bad dyn_mode");
  const bool has_dyn = b->dyn_mode != FOT_DYN_NONE && (long long)b->S * b->P * b->T_obs > 0;
  if (has_dyn && !b->dyn) return fail(FOT_ERR_ARG, "fot_assess_trajectories: dynamic obstacles missing");
  if ((size_t)b->n_q * a->m * a->n_r > 0x7fffffffull) return fail(FOT_ERR_ARG, "fot_assess_trajectories: batch too large");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  // one sample per thread; a whole trajectory always fits (n_t <= FOT_MAX_ASSESS_NT <= kAssessMaxThreads)
  const int samples = (int)std::min<long long>((long long)a->m * a->n_t, kAssessMaxThreads);
  const int threads = std::max(64, (std::max(samples, a->n_t) + 31) / 32 * 32);
  const size_t smem = (size_t)threads * assess_smem_per_thread(std::max(h->plan.cfg.n_circles, 1));
  // the kernel's static arrays (7.3 KB) count against the 48 KB a launch gets without opting in
  if (smem > 32 * 1024) CK(cudaFuncSetAttribute(fot_assess, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  Batch B{};
  B.n_q = b->n_q;
  B.n_static = b->n_static; B.static_per_query = b->static_per_query;
  B.S = has_dyn ? b->S : 0; B.P = has_dyn ? b->P : 0; B.T_obs = has_dyn ? b->T_obs : 0; B.dyn_mode = b->dyn_mode;
  B.dyn_raw = has_dyn ? b->dyn : nullptr;
  B.static_raw = b->n_static > 0 ? b->static_obs : nullptr;
  const Assess A{a->m, a->n_t, a->n_r, a->series, a->len, a->r2, a->dyn_min, a->dyn_at, a->static_min, a->static_at,
                 a->dyn_hits, a->first_hit, a->static_hit};
  fot_assess<<<(unsigned)b->n_q, threads, smem, st>>>(h->plan, B, A);
  CK(cudaGetLastError());
  if (!stream) CK(cudaStreamSynchronize(st));
  return FOT_OK;
}

extern "C" int fot_assess_candidates(fot_handle_t* h, const fot_batch_t* b, const fot_batch_t* f, int cand_stride,
                                     const fot_assessed_t* a, int32_t* keep, void* stream) {
  if (!h || !b || !f || !a) return fail(FOT_ERR_ARG, "fot_assess_candidates: null argument");
  if (b->n_q < 1 || b->n_v_max < 1) return fail(FOT_ERR_ARG, "fot_assess_candidates: n_q and n_v_max must be >= 1");
  if (a->series || a->len) return fail(FOT_ERR_ARG, "fot_assess_candidates: series and len must be null (candidates are regenerated)");
  if (a->m != cand_stride) return fail(FOT_ERR_ARG, "fot_assess_candidates: m must equal cand_stride");
  if (a->n_r < 1 || a->n_r > FOT_MAX_RADII) return fail(FOT_ERR_ARG, "fot_assess_candidates: n_r must be in [1, FOT_MAX_RADII]");
  if (!a->r2) return fail(FOT_ERR_ARG, "fot_assess_candidates: null r2");
  if (!a->dyn_min || !a->dyn_at || !a->static_min || !a->static_at || !a->dyn_hits || !a->first_hit || !a->static_hit)
    return fail(FOT_ERR_ARG, "fot_assess_candidates: null output array");
  if (!b->frenet || !b->target_speed || !b->v_grid || !b->n_v) return fail(FOT_ERR_ARG, "fot_assess_candidates: null query array");
  if (f->n_static < 0 || f->S < 0 || f->P < 0 || f->T_obs < 0)
    return fail(FOT_ERR_ARG, "fot_assess_candidates: negative obstacle shape");
  if (f->n_static > 0 && !f->static_obs) return fail(FOT_ERR_ARG, "fot_assess_candidates: static obstacles missing");
  if (f->dyn_mode != FOT_DYN_NONE && f->dyn_mode != FOT_DYN_SINGLE && f->dyn_mode != FOT_DYN_DISTRIBUTION)
    return fail(FOT_ERR_ARG, "fot_assess_candidates: bad dyn_mode");
  const bool has_dyn = f->dyn_mode != FOT_DYN_NONE && (long long)f->S * f->P * f->T_obs > 0;
  if (has_dyn && !f->dyn) return fail(FOT_ERR_ARG, "fot_assess_candidates: dynamic obstacles missing");
  if ((size_t)b->n_q * cand_stride * a->n_r > 0x7fffffffull) return fail(FOT_ERR_ARG, "fot_assess_candidates: batch too large");
  const int n_max = fot_candidate_count(h, b->n_v_max, 1);
  if (cand_stride < n_max) return fail(FOT_ERR_ARG, "fot_assess_candidates: cand_stride too small");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  Batch B{};
  B.n_q = b->n_q; B.n_v_max = b->n_v_max;
  B.frenet = b->frenet; B.target = b->target_speed; B.v_grid = b->v_grid; B.n_v = b->n_v;
  B.n_static = f->n_static; B.static_per_query = f->static_per_query;
  B.S = has_dyn ? f->S : 0; B.P = has_dyn ? f->P : 0; B.T_obs = has_dyn ? f->T_obs : 0; B.dyn_mode = f->dyn_mode;
  B.dyn_raw = has_dyn ? f->dyn : nullptr;
  B.static_raw = f->n_static > 0 ? f->static_obs : nullptr;
  B.rt = routes_of(h, 0);
  AssessCand C{};
  C.A = Assess{a->m, 0, a->n_r, nullptr, nullptr, a->r2, a->dyn_min, a->dyn_at, a->static_min, a->static_at,
               a->dyn_hits, a->first_hit, a->static_hit};
  C.keep = keep;
  const long long SP = (long long)B.S * B.P;
  if (has_dyn) {
    // one bit per pedestrian trajectory: a NaN at any step (the NaN rule), once per launch
    C.nan_words = (int32_t)((SP + 31) / 32);
    const long long n_words = (long long)b->n_q * C.nan_words;
    if ((n_words * 32 + 255) / 256 > 0x7fffffffll) return fail(FOT_ERR_ARG, "fot_assess_candidates: field too large for one launch");
    CK(h->ca_nan.reserve((size_t)n_words * sizeof(unsigned)));
    C.nan_bits = (const unsigned*)h->ca_nan.p;
    fot_assess_cand_nan<<<(unsigned)((n_words * 32 + 255) / 256), 256, 0, st>>>((const double2*)f->dyn, SP, B.T_obs, n_words,
                                                                             C.nan_words, (unsigned*)h->ca_nan.p);
  }
  C.sc = has_dyn ? std::min(B.S, kCandPass) : 0;
  // CTAs per query: one once the batch fills the GPU several times over; a small batch (one plan() call of 66 563
  // candidates) is dealt to many
  const long long per_cta = kCandThreads;
  long long cpq = ((long long)h->sms * 4 + b->n_q - 1) / b->n_q;
  cpq = std::max<long long>(1, std::min<long long>(cpq, (n_max + per_cta - 1) / per_cta));
  C.cpq = (int32_t)cpq;
  if ((long long)b->n_q * cpq > 0x7fffffffll) return fail(FOT_ERR_ARG, "fot_assess_candidates: batch too large for one launch");
  const size_t stage_bytes = (size_t)SP * B.T_obs * sizeof(double2);
  const bool stage = has_dyn && stage_bytes <= kCandStageMax;
  const size_t smem = assess_cand_smem(h->plan.n_t_max, a->n_r, C.sc, stage ? stage_bytes : 0);
  if (smem > (size_t)h->smem_optin) return fail(FOT_ERR_TOO_LARGE, "fot_assess_candidates: shared memory");
  auto kern = stage ? fot_assess_cand<true> : fot_assess_cand<false>;
  if (smem > 32 * 1024) CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)(b->n_q * cpq), kCandThreads, smem, st>>>(h->plan, B, C);
  CK(cudaGetLastError());
  if (!stream) CK(cudaStreamSynchronize(st));
  return FOT_OK;
}

// The query arrays the cost pieces read, as a Batch; and the pieces themselves into the handle's scratch, on `st`.
static int weighted_pieces(fot_handle* h, const fot_batch_t* b, cudaStream_t st, Batch* B) {
  *B = Batch{};
  B->n_q = b->n_q; B->n_v_max = b->n_v_max;
  B->frenet = b->frenet; B->target = b->target_speed; B->v_grid = b->v_grid; B->n_v = b->n_v;
  B->rt = routes_of(h, 0);
  const long long n_prof = (long long)b->n_q * piece_profiles(h->plan.cfg, b->n_v_max);
  if ((n_prof + 255) / 256 > 0x7fffffffll) return fail(FOT_ERR_ARG, "batch too large for one launch");
  CK(h->w_pieces.reserve((size_t)b->n_q * piece_stride(h->plan.cfg, b->n_v_max) * sizeof(double)));
  fot_cost_pieces<<<(unsigned)((n_prof + 255) / 256), 256, (size_t)kTT * h->plan.n_t_max * sizeof(double), st>>>(
      h->plan, *B, (double*)h->w_pieces.p);
  return FOT_OK;
}

extern "C" int fot_select_weighted(fot_handle_t* h, const fot_batch_t* b, const uint8_t* cand_cat, int cand_stride,
                                   const fot_weighted_t* out, void* stream) {
  if (!h || !b || !out || !cand_cat) return fail(FOT_ERR_ARG, "fot_select_weighted: null argument");
  if (b->n_q < 1 || b->n_v_max < 1) return fail(FOT_ERR_ARG, "fot_select_weighted: n_q and n_v_max must be >= 1");
  if (out->n_w < 1 || out->n_w > FOT_MAX_WEIGHT_SETS)
    return fail(FOT_ERR_ARG, "fot_select_weighted: n_w must be in [1, FOT_MAX_WEIGHT_SETS]");
  if (out->per_query != 0 && out->per_query != 1) return fail(FOT_ERR_ARG, "fot_select_weighted: per_query must be 0 or 1");
  if (!out->weights || !out->idx || !out->cost) return fail(FOT_ERR_ARG, "fot_select_weighted: null weights, idx or cost");
  if (out->series && !out->len) return fail(FOT_ERR_ARG, "fot_select_weighted: series needs len");
  if (cand_stride < fot_candidate_count(h, b->n_v_max, 1)) return fail(FOT_ERR_ARG, "fot_select_weighted: cand_stride too small");
  if (!b->frenet || !b->target_speed || !b->v_grid || !b->n_v) return fail(FOT_ERR_ARG, "fot_select_weighted: null query array");
  const size_t n_chunks = ((size_t)out->n_w + kWChunk - 1) / kWChunk;
  if ((size_t)b->n_q * n_chunks > 0x7fffffffull || (size_t)b->n_q * out->n_w > 0x7fffffffull)
    return fail(FOT_ERR_ARG, "fot_select_weighted: batch too large for one launch");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  Batch B;
  int rc = weighted_pieces(h, b, st, &B);
  if (rc != FOT_OK) return rc;
  const Weighted W{out->n_w, out->per_query, out->weights, out->idx, out->cost, out->len};
  fot_select_weighted_kernel<<<(unsigned)((size_t)b->n_q * n_chunks), kWThreads, 0, st>>>(
      h->plan, B, cand_cat, cand_stride, (const double*)h->w_pieces.p, W);
  if (out->len) {
    // the selected candidates' series, regenerated as fot_winner does: a ranked list of n_w entries per query
    const Ranked R{out->n_w, out->idx, out->cost, out->len, out->series};
    fot_rank_series<<<(unsigned)((size_t)b->n_q * out->n_w), 128, (size_t)kTT * h->plan.n_t_max * sizeof(double), st>>>(h->plan, B, R);
  }
  CK(cudaGetLastError());
  if (!stream) CK(cudaStreamSynchronize(st));
  return FOT_OK;
}

extern "C" int fot_cost_terms(fot_handle_t* h, const fot_batch_t* b, int cand_stride, double* terms, void* stream) {
  if (!h || !b || !terms) return fail(FOT_ERR_ARG, "fot_cost_terms: null argument");
  if (b->n_q < 1 || b->n_v_max < 1) return fail(FOT_ERR_ARG, "fot_cost_terms: n_q and n_v_max must be >= 1");
  if (cand_stride < fot_candidate_count(h, b->n_v_max, 1)) return fail(FOT_ERR_ARG, "fot_cost_terms: cand_stride too small");
  if (!b->frenet || !b->target_speed || !b->v_grid || !b->n_v) return fail(FOT_ERR_ARG, "fot_cost_terms: null query array");
  const long long n = (long long)b->n_q * cand_stride;
  if ((n + 255) / 256 > 0x7fffffffll) return fail(FOT_ERR_ARG, "fot_cost_terms: batch too large for one launch");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  Batch B;
  int rc = weighted_pieces(h, b, st, &B);
  if (rc != FOT_OK) return rc;
  fot_cost_terms_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h->plan, B, cand_stride, (const double*)h->w_pieces.p, terms);
  CK(cudaGetLastError());
  if (!stream) CK(cudaStreamSynchronize(st));
  return FOT_OK;
}

// First k samples of every winner series, packed [n][FOT_N_SERIES][k] (fot_result_t.winner_samples): a strided copy of
// 16-byte rows is slow on the copy engines, a contiguous one is not.
__global__ void fot_pack_heads(const double* __restrict__ winner, double* __restrict__ heads, long long n_rows, int NT, int k) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rows * k) return;
  const long long row = i / k;
  heads[i] = winner[row * NT + (i - row * k)];
}

// Read-back of one chunk's winner block into the caller's arrays on stream `ds` (after `st`'s kernels).
static int read_back(fot_handle* h, const fot_result_t* r, const fot_result_t& dr, double* heads_d, int q0, int cq, int NT,
                     cudaStream_t st, cudaStream_t ds, cudaEvent_t done) {
  const int k = r->winner_samples > 0 ? std::min(r->winner_samples, NT) : 0;
  if (k > 0) {
    const long long n_rows = (long long)cq * FOT_N_SERIES;
    fot_pack_heads<<<(unsigned)((n_rows * k + 255) / 256), 256, 0, st>>>(dr.winner, heads_d, n_rows, NT, k);
  }
  CK(cudaEventRecord(done, st));
  CK(cudaStreamWaitEvent(ds, done, 0));
  CK(cudaMemcpyAsync(r->best_idx + q0, dr.best_idx, (size_t)cq * 4, cudaMemcpyDeviceToHost, ds));
  CK(cudaMemcpyAsync(r->best_cost + q0, dr.best_cost, (size_t)cq * 8, cudaMemcpyDeviceToHost, ds));
  CK(cudaMemcpyAsync(r->stats + (size_t)q0 * FOT_N_STATS, dr.stats, (size_t)cq * FOT_N_STATS * 4, cudaMemcpyDeviceToHost, ds));
  CK(cudaMemcpyAsync(r->winner_len + q0, dr.winner_len, (size_t)cq * 4, cudaMemcpyDeviceToHost, ds));
  if (k > 0)
    CK(cudaMemcpyAsync(r->winner + (size_t)q0 * FOT_N_SERIES * k, heads_d, (size_t)cq * FOT_N_SERIES * k * 8, cudaMemcpyDeviceToHost, ds));
  else
    CK(cudaMemcpyAsync(r->winner + (size_t)q0 * FOT_N_SERIES * NT, dr.winner, (size_t)cq * FOT_N_SERIES * NT * 8,
                       cudaMemcpyDeviceToHost, ds));
  if (r->cand_cat)
    CK(cudaMemcpyAsync(r->cand_cat + (size_t)q0 * r->cand_stride, dr.cand_cat, (size_t)cq * r->cand_stride,
                       cudaMemcpyDeviceToHost, ds));
  if (r->cand_cost)
    CK(cudaMemcpyAsync(r->cand_cost + (size_t)q0 * r->cand_stride, dr.cand_cost, (size_t)cq * r->cand_stride * 8,
                       cudaMemcpyDeviceToHost, ds));
  return FOT_OK;
}

// A failed multi-chunk call may leave earlier chunks in flight: kernels, upload slices and read-backs into the
// CALLER's result arrays, and (gated mode) CTAs spinning on slice flags that will never be written.  Nothing of that
// may still be running when the error is reported -- the caller is free to release its arrays, and the next call
// reuses the handle's scratch and gate flags.  Releases the waiting CTAs (their results are discarded), waits for
// every stream of the handle and clears the gate error word; keeps the error text of the failure.
static void drain_after_failure(fot_handle* h) {
  const std::string keep = g_err;
  if (h->gate_d.p && h->gate_epoch) {
    std::vector<uint32_t> w(kGateSlices, h->gate_epoch);
    cudaMemcpy(h->gate_d.p, w.data(), kGateSlices * sizeof(uint32_t), cudaMemcpyHostToDevice);
  }
  for (cudaStream_t s : {h->copy_stream, h->stream, h->stream2, h->pstream[0], h->pstream[1], h->pstream[2], h->pstream[3],
                         h->d2h_stream})
    if (s) cudaStreamSynchronize(s);
  if (h->gate_d.p) cudaMemset((uint32_t*)h->gate_d.p + kGateSlices, 0, sizeof(uint32_t));
  cudaGetLastError();
  g_err = keep;
}

// device-side span of a call that ran on several streams (fot_last_kernel_ms): `first` carries ev0; ev1 is recorded
// on it after every other stream of the handle has been joined
static int close_span(fot_handle* h, cudaStream_t first) {
  for (cudaStream_t s : {h->stream, h->stream2, h->pstream[0], h->pstream[1], h->pstream[2], h->pstream[3]}) {
    if (s == first) continue;
    CK(cudaEventRecord(h->ev_join, s));
    CK(cudaStreamWaitEvent(first, h->ev_join, 0));
  }
  CK(cudaEventRecord(h->ev1, first));
  return FOT_OK;
}

// Query ranges of a host-result call: range c is queries [bound[c], bound[c + 1]).  gated (host-pointer call only): the
// sweep waits for slices of the obstacle upload, not for whole ranges.
struct Ranges {
  int n = 1;
  int bound[fot_handle::kMaxChunks + 1] = {};
  bool gated = false;
};

// Ranges ending at about frac16[i] / 16 of the nq queries, in whole waves of the sweep (one CTA per query, two CTAs per
// SM) where possible, and a last range ending at nq.
static void cut16(const fot_handle* h, int nq, std::initializer_list<int> frac16, Ranges* rg) {
  const int wave = 2 * h->sms;
  rg->n = 0;
  rg->bound[0] = 0;
  for (int f : frac16) {
    const int cut = std::max(1, (int)((long long)nq * f / 16 / wave)) * wave;
    rg->bound[rg->n + 1] = std::min(nq, std::max(cut, rg->bound[rg->n]));
    ++rg->n;
  }
  rg->bound[++rg->n] = nq;
}

static Ranges plan_ranges(const fot_handle* h, const fot_batch_t* b, bool host) {
  const int nq = b->n_q;
  const bool has_dyn = b->dyn_mode != FOT_DYN_NONE;
  Ranges rg;
  rg.bound[1] = nq;
  const std::string keep = g_err;      // a kernel the probe below refuses is not an error of this call
  if (host) {
    // Ranges only pay when the obstacle upload is large.  The kernels are the longer leg of the pipeline (the upload runs
    // at PCIe speed), so the first ranges are small -- the sweep starts after 1/16 of the upload -- and the rest large
    // enough to keep the wave tail short: about 1/16, 1/8, 3/16, 5/16, 5/16 of the queries.
    const size_t upload = has_dyn ? (size_t)nq * b->S * b->P * b->T_obs * 16 : 0;
    if (upload > ((size_t)8 << 20) && nq >= 1024) cut16(h, nq, {1, 3, 6, 11}, &rg);
    if (h->opt.host_chunks > 0) {
      rg.n = std::max(1, std::min(fot_handle::kMaxChunks, h->opt.host_chunks));
      const int per = (nq + rg.n - 1) / rg.n;
      for (int c = 0; c <= rg.n; ++c) rg.bound[c] = std::min(nq, c * per);
    }
    // Gated, the sweep does not wait for whole ranges, so a few large ones do: about 1/2, 5/16, 3/16 of the queries.
    Sweep s;
    rg.gated = h->opt.gated && rg.n > 1 && has_dyn && nq < (1 << 22) && select_sweep(h, b, true, &s) == FOT_OK;
    if (rg.gated && h->opt.host_chunks <= 0) cut16(h, nq, {8, 13}, &rg);
  } else if (nq >= 1024) {
    cut16(h, nq, {8, 13}, &rg);
  }
  g_err = keep;
  return rg;
}

// FOT_DEBUG_TIMING=1: the device timeline of a host-pointer call on stderr, in ms from the start of the call
// (profiles/r1/e2e_timeline.txt; tools/tuning/e2e_lib.sh reads the last lines).  A timeline that is off records nothing.
struct Timeline {
  enum { kStart, kCopyStart, kCopiesDone, kKernelsDone, kRange };   // then per range: upload done,
  static constexpr int kEvents = kRange + 4 * fot_handle::kMaxChunks;  // kernels start / end, read-back done
  cudaEvent_t ev[kEvents] = {};
  bool marked[kEvents] = {};
  explicit Timeline(bool on) { if (on) for (auto& e : ev) cudaEventCreate(&e); }
  ~Timeline() { for (auto e : ev) if (e) cudaEventDestroy(e); }
  void mark(int i, cudaStream_t s) { if (ev[i]) marked[i] = cudaEventRecord(ev[i], s) == cudaSuccess; }
  void range(int c, int k, cudaStream_t s) { mark(kRange + 4 * c + k, s); }
  float ms(int i) const {
    float t = -1.0f;
    if (marked[kStart] && marked[i] && cudaEventSynchronize(ev[kStart]) == cudaSuccess && cudaEventSynchronize(ev[i]) == cudaSuccess)
      cudaEventElapsedTime(&t, ev[kStart], ev[i]);
    return t;
  }
  void print(const Ranges& rg) const {
    if (!ev[kStart]) return;
    fprintf(stderr, "[fot] chunks=%d copy-stream start %.3f ms, copies done %.3f ms, first kernel may start %.3f ms, kernels done %.3f ms\n",
            rg.n, ms(kCopyStart), ms(kCopiesDone), ms(kRange + 1), ms(kKernelsDone));   // range 0 is never empty
    for (int c = 0; c < rg.n; ++c) {
      const int e = kRange + 4 * c;
      fprintf(stderr, "[fot]   chunk %2d queries %5d..%5d  upload done %.3f  kernels %.3f -> %.3f  read-back done %.3f\n", c,
              rg.bound[c], rg.bound[c + 1], ms(e), ms(e + 1), ms(e + 2), ms(e + 3));
    }
  }
};

// The range loop of both host-result calls: `b` is the whole batch in device memory, `r` the caller's host arrays.  Range c
// is swept once wait[c] (if given) has fired, and its winners go back on the d2h stream as soon as its kernels finish, so
// only the last range's read-back is exposed.  With `prio` the ranges run on streams of descending priority: every
// range's kernels are eligible from the start, and a CTA of a later range that got an SM slot early would only sit there
// waiting (gated: for its slice of the upload).  Otherwise they alternate two compute streams, so that the next range's
// CTAs fill the SMs the tail wave of the previous range leaves idle (the ranges touch disjoint scratch, see launch_all).
static int run_ranges(fot_handle* h, const fot_batch_t* b, const fot_result_t* r, const Ranges& rg, Gate gate, bool prio,
                      const cudaEvent_t* wait, Timeline& tl) {
  const int nq = b->n_q, NT = h->plan.n_t_max;
  size_t ro = 0;
  auto rtake = [&](size_t bytes) { size_t o = ro; ro = align_up(ro + bytes); return o; };
  const size_t r_bi = rtake((size_t)nq * 4), r_bc = rtake((size_t)nq * 8), r_st = rtake((size_t)nq * FOT_N_STATS * 4),
               r_wl = rtake((size_t)nq * 4), r_w = rtake((size_t)nq * FOT_N_SERIES * NT * 8);
  const size_t r_cc = r->cand_cat ? rtake((size_t)nq * r->cand_stride) : 0;
  const size_t r_cs = r->cand_cost ? rtake((size_t)nq * r->cand_stride * 8) : 0;
  const int k_head = r->winner_samples > 0 ? std::min(r->winner_samples, NT) : 0;
  const size_t r_wh = k_head ? rtake((size_t)nq * FOT_N_SERIES * k_head * 8) : 0;
  CK(h->out_d.reserve(ro));
  char* od = (char*)h->out_d.p;
  h->last_winner_d = (const double*)(od + r_w);     // fot_fetch_winners
  h->last_winner_nq = nq;
  const size_t dyn_q_bytes = b->dyn_mode != FOT_DYN_NONE ? (size_t)b->S * b->P * b->T_obs * 16 : 0;
  auto stream_of = [&](int i) { return prio ? h->pstream[i & 3] : (i & 1) ? h->stream2 : h->stream; };
  int n_issued = 0;
  for (int c = 0; c < rg.n; ++c) {
    const int q0 = rg.bound[c], cq = rg.bound[c + 1] - q0;
    if (cq <= 0) continue;
    const int i = n_issued++;
    cudaStream_t st = stream_of(i);
    if (wait) CK(cudaStreamWaitEvent(st, wait[c], 0));
    if (i == 0) CK(cudaEventRecord(h->ev0, st));
    tl.range(c, 1, st);
    fot_batch_t db = *b;
    db.n_q = cq;
    db.frenet = b->frenet + (size_t)q0 * 6;
    db.target_speed = b->target_speed + q0;
    db.limits = b->limits + (size_t)q0 * 4;
    db.stop_dist = b->stop_dist + q0;
    db.v_grid = b->v_grid + (size_t)q0 * b->n_v_max;
    db.n_v = b->n_v + q0;
    if (dyn_q_bytes) db.dyn = (const double*)((const char*)b->dyn + (size_t)q0 * dyn_q_bytes);
    if (b->n_static > 0 && b->static_per_query) db.static_obs = b->static_obs + (size_t)q0 * b->n_static * 2;
    fot_result_t dr = *r;
    dr.best_idx = (int32_t*)(od + r_bi) + q0;
    dr.best_cost = (double*)(od + r_bc) + q0;
    dr.stats = (int32_t*)(od + r_st) + (size_t)q0 * FOT_N_STATS;
    dr.winner_len = (int32_t*)(od + r_wl) + q0;
    dr.winner = (double*)(od + r_w) + (size_t)q0 * FOT_N_SERIES * NT;
    dr.cand_cat = r->cand_cat ? (uint8_t*)(od + r_cc) + (size_t)q0 * r->cand_stride : nullptr;
    dr.cand_cost = r->cand_cost ? (double*)(od + r_cs) + (size_t)q0 * r->cand_stride : nullptr;
    int rc = launch_all(h, &db, &dr, st, (size_t)q0, (size_t)nq, gate, /*record_span=*/false);
    if (rc != FOT_OK) return rc;
    tl.range(c, 2, st);
    // on their own stream, so that the next range's kernels never queue behind a copy engine busy with the uploads
    rc = read_back(h, r, dr, (double*)(od + r_wh) + (size_t)q0 * FOT_N_SERIES * k_head, q0, cq, NT, st, h->d2h_stream, h->ev_done[c]);
    if (rc != FOT_OK) return rc;
    tl.range(c, 3, h->d2h_stream);
  }
  const int rc = close_span(h, stream_of(0));
  if (rc != FOT_OK) return rc;
  tl.mark(Timeline::kKernelsDone, stream_of(0));
  CK(cudaStreamSynchronize(h->d2h_stream));   // the last read-backs wait for the last kernels of every compute stream
  for (int i = 0; i < n_issued && i < 4; ++i) CK(cudaStreamSynchronize(stream_of(i)));
  tl.print(rg);
  return FOT_OK;
}

// Host-pointer entry point.  Small per-query arrays go through one pinned blob; the obstacle tensor is copied straight
// from the caller's memory (pinned memory makes that a true async DMA).  A large upload is pipelined with the sweep: the
// sweep either waits for fine slices of it (gated) or for whole ranges of queries, so that range c+1's upload runs on
// the copy stream while range c's kernels run.
static int plan_batch_host_impl(fot_handle_t* h, const fot_batch_t* b, const fot_result_t* r) {
  const int nq = b->n_q;
  // ---- small per-query arrays: one pinned blob, one H2D -------------------------------
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
  const size_t o_fr = take((size_t)nq * 6 * 8), o_tg = take((size_t)nq * 8), o_lm = take((size_t)nq * 4 * 8),
               o_sd = take((size_t)nq * 8), o_vg = take((size_t)nq * b->n_v_max * 8), o_nv = take((size_t)nq * 4);
  CK(h->stage_h.reserve(off));
  CK(h->stage_d.reserve(off));
  char* sh = (char*)h->stage_h.p;
  memcpy(sh + o_fr, b->frenet, (size_t)nq * 6 * 8);
  memcpy(sh + o_tg, b->target_speed, (size_t)nq * 8);
  memcpy(sh + o_lm, b->limits, (size_t)nq * 4 * 8);
  memcpy(sh + o_sd, b->stop_dist, (size_t)nq * 8);
  memcpy(sh + o_vg, b->v_grid, (size_t)nq * b->n_v_max * 8);
  memcpy(sh + o_nv, b->n_v, (size_t)nq * 4);
  // The compute stream carries kernels and event records only: every copy runs on the copy / d2h
  // streams.  (A copy on the compute stream makes the driver service that stream's later timed event
  // records on the copy engine, where they queue behind the uploads and serialise the pipeline.)
  CK(cudaMemcpyAsync(h->stage_d.p, sh, off, cudaMemcpyHostToDevice, h->copy_stream));
  const char* sd = (const char*)h->stage_d.p;
  const bool has_dyn = b->dyn_mode != FOT_DYN_NONE;
  const size_t dyn_q_bytes = has_dyn ? (size_t)b->S * b->P * b->T_obs * 16 : 0;
  if (has_dyn) CK(h->dyn_d.reserve((size_t)nq * dyn_q_bytes));
  if (b->n_static > 0) {
    const size_t bytes = (size_t)(b->static_per_query ? nq : 1) * b->n_static * 16;
    CK(h->stat_d.reserve(bytes));
    CK(cudaMemcpyAsync(h->stat_d.p, b->static_obs, bytes, cudaMemcpyHostToDevice, h->copy_stream));
  }
  // the batch as the kernels read it
  fot_batch_t db = *b;
  db.frenet = (const double*)(sd + o_fr);
  db.target_speed = (const double*)(sd + o_tg);
  db.limits = (const double*)(sd + o_lm);
  db.stop_dist = (const double*)(sd + o_sd);
  db.v_grid = (const double*)(sd + o_vg);
  db.n_v = (const int32_t*)(sd + o_nv);
  if (has_dyn) db.dyn = (const double*)h->dyn_d.p;
  if (b->n_static > 0) db.static_obs = (const double*)h->stat_d.p;
  const Ranges rg = plan_ranges(h, b, true);
  // Gated: the upload is cut into fine slices, each followed by a 4-byte write that publishes "queries uploaded so
  // far", and every CTA of the sweep waits for its own query's slice (ItemGeom::gate).
  int n_up = 0, ub[kGateSlices + 1] = {0};
  Gate gate{};
  if (rg.gated) {
    const bool fresh = h->gate_d.p == nullptr;
    CK(h->gate_d.reserve((kGateSlices + 1) * sizeof(uint32_t)));
    CK(h->gate_h.reserve((kGateSlices + 1) * sizeof(uint32_t)));
    if (fresh) CK(cudaMemset(h->gate_d.p, 0, (kGateSlices + 1) * sizeof(uint32_t)));
    if (++h->gate_epoch == 0) h->gate_epoch = 1;             // 0 is the value of a fresh flag
    gate.word = (unsigned*)h->gate_d.p;
    gate.epoch = h->gate_epoch;
    n_up = std::max(1, std::min(kGateSlices, h->opt.gate_uploads));
    gate.per = (nq + n_up - 1) / n_up;
    n_up = (nq + gate.per - 1) / gate.per;
    for (int u = 0; u <= n_up; ++u) ub[u] = std::min(nq, u * gate.per);
  }
  const auto t_wall0 = std::chrono::steady_clock::now();
  Timeline tl(h->opt.debug_timing != 0);
  tl.mark(Timeline::kStart, h->stream);
  tl.mark(Timeline::kCopyStart, h->copy_stream);
  CK(cudaEventRecord(h->ev_blob, h->copy_stream));
  // every obstacle upload is queued first (they depend on nothing)
  if (rg.gated) {
    // each slice is followed on the upload stream by the write of its flag, which stream order keeps behind the slice
    uint32_t* words = (uint32_t*)h->gate_h.p;
    for (int u = 0; u < n_up; ++u) {
      const int q0 = ub[u], cq = ub[u + 1] - q0;
      if (cq <= 0) continue;
      char* dst = (char*)h->dyn_d.p + (size_t)q0 * dyn_q_bytes;
      const char* src = (const char*)b->dyn + (size_t)q0 * dyn_q_bytes;
      CK(cudaMemcpyAsync(dst, src, (size_t)cq * dyn_q_bytes, cudaMemcpyHostToDevice, h->copy_stream));
      words[u] = gate.epoch;
      if (StreamWrite32 wr = h->opt.gate_memcpy ? nullptr : stream_write32()) {
        if (wr(h->copy_stream, (unsigned long long)(uintptr_t)(gate.word + u), gate.epoch, 0u) != 0)
          return fail(FOT_ERR_CUDA, "cuStreamWriteValue32");
      } else {
        CK(cudaMemcpyAsync(gate.word + u, words + u, sizeof(uint32_t), cudaMemcpyHostToDevice, h->copy_stream));
      }
    }
  } else if (has_dyn)
    for (int c = 0; c < rg.n; ++c) {
      const int q0 = rg.bound[c], cq = rg.bound[c + 1] - q0;
      if (cq <= 0) continue;
      char* dst = (char*)h->dyn_d.p + (size_t)q0 * dyn_q_bytes;
      const char* src = (const char*)b->dyn + (size_t)q0 * dyn_q_bytes;
      CK(cudaMemcpyAsync(dst, src, (size_t)cq * dyn_q_bytes, cudaMemcpyHostToDevice, h->copy_stream));
      CK(cudaEventRecord(h->ev_copy[c], h->copy_stream));
      tl.range(c, 0, h->copy_stream);
    }
  tl.mark(Timeline::kCopiesDone, h->copy_stream);
  if (h->opt.debug_timing) {
    cudaPointerAttributes pa{};
    cudaError_t pe = cudaPointerGetAttributes(&pa, b->dyn);
    fprintf(stderr, "[fot] dyn pointer attr: err=%d type=%d (0 unregistered, 1 host, 2 device, 3 managed)\n", (int)pe, (int)pa.type);
  }
  cudaEvent_t wait[fot_handle::kMaxChunks];
  for (int c = 0; c < rg.n; ++c) wait[c] = has_dyn && !rg.gated ? h->ev_copy[c] : h->ev_blob;
  const int rc = run_ranges(h, &db, r, rg, gate, /*prio=*/rg.gated, wait, tl);
  if (rc != FOT_OK) return rc;
  if (!rg.gated) return FOT_OK;
  CK(cudaStreamSynchronize(h->copy_stream));
  if (std::chrono::steady_clock::now() - t_wall0 > std::chrono::nanoseconds(kGateTimeoutNs)) {
    unsigned gave_up = 0;
    CK(cudaMemcpy(&gave_up, gate.word + kGateSlices, sizeof(unsigned), cudaMemcpyDeviceToHost));
    if (gave_up) {
      cudaMemset(gate.word + kGateSlices, 0, sizeof(unsigned));
      return fail(FOT_ERR_CUDA, "gated sweep: the obstacle upload did not arrive");
    }
  }
  return FOT_OK;
}

extern "C" int fot_plan_batch_host(fot_handle_t* h, const fot_batch_t* b, const fot_result_t* r) {
  int rc = check_batch(h, b, r);
  if (rc != FOT_OK) return rc;
  CK(cudaSetDevice(h->device));
  rc = plan_batch_host_impl(h, b, r);
  if (rc != FOT_OK) drain_after_failure(h);
  return rc;
}

// Device inputs, HOST results: the call of a caller whose obstacle tensor was produced on the GPU (the prediction
// post-processing of fot_predict.cuh) but who consumes the winners on the host.  Large batches are swept in three
// ranges on the priority streams, and each range's winners go back over PCIe while the next range is swept, so only
// the last range's read-back is exposed.  `stream` is the stream on which the inputs become ready (NULL: they are
// ready now).  Returns when the results are in `res`.
extern "C" int fot_plan_batch_device_to_host(fot_handle_t* h, const fot_batch_t* b, const fot_result_t* r, void* stream) {
  int rc = check_batch(h, b, r);
  if (rc != FOT_OK) return rc;
  CK(cudaSetDevice(h->device));
  cudaEvent_t wait[fot_handle::kMaxChunks];
  for (auto& e : wait) e = h->ev_blob;
  if (stream) CK(cudaEventRecord(h->ev_blob, (cudaStream_t)stream));
  Timeline off(false);
  rc = run_ranges(h, b, r, plan_ranges(h, b, false), Gate{}, /*prio=*/true, stream ? wait : nullptr, off);
  if (rc != FOT_OK) drain_after_failure(h);
  return rc;
}

// ---- the gather of a sharded sweep over peer memory ---------------------------------------------------------------
extern "C" int fot_set_result_mirror(fot_handle_t* h, const fot_result_t* mirror, void* flag) {
  if (!h) return fail(FOT_ERR_ARG, "fot_set_result_mirror: null handle");
  if (!mirror) { h->mirror = fot_result_t{}; h->mirror_flag = nullptr; h->mirror_seq = 0; return FOT_OK; }
  if (!mirror->best_idx || !mirror->best_cost || !mirror->stats || !mirror->winner_len || !mirror->winner)
    return fail(FOT_ERR_ARG, "fot_set_result_mirror: null mirror array");
  h->mirror = *mirror;
  if ((unsigned*)flag != h->mirror_flag) h->mirror_seq = 0;     // a new flag word starts a new sequence: 1, 2, 3, ...
  h->mirror_flag = (unsigned*)flag;
  return FOT_OK;
}

// ---- routes: per-query reference paths (DESIGN.md section 4h) ------------------------------------------------------
extern "C" int fot_add_route(fot_handle_t* h, const fot_route_t* route, int32_t* route_id) {
  if (!h || !route || !route_id) return fail(FOT_ERR_ARG, "fot_add_route: null argument");
  const int nx = route->nx;
  if (nx < 2) return fail(FOT_ERR_ARG, "fot_add_route: a route needs at least 2 knots");
  const double* tabs[9] = {route->knots, route->xa, route->xb, route->xc, route->xd, route->ya, route->yb, route->yc, route->yd};
  for (const double* t : tabs)
    if (!t) return fail(FOT_ERR_ARG, "fot_add_route: null spline table");
  if (h->rt_tab.size() + 9 * (size_t)nx > 0x7fffffffull) return fail(FOT_ERR_TOO_LARGE, "fot_add_route: route tables beyond 2^31 doubles");
  // host copies first; the device blob is rebuilt from them (a new route is rare, and never on the planning path)
  std::vector<double> tab = h->rt_tab;
  const size_t off = tab.size();
  for (int k = 0; k < 9; ++k) {
    const int n = (k == 2 || k == 4 || k == 6 || k == 8) ? nx - 1 : nx;     // b and d have nx - 1 entries
    tab.insert(tab.end(), tabs[k], tabs[k] + n);
    if (n < nx) tab.push_back(0.0);
  }
  std::vector<int32_t> nxs = h->rt_nx, offs = h->rt_off;
  nxs.push_back(nx);
  nxs[0] = (int32_t)(nxs.size() - 1);
  offs.push_back((int32_t)off);
  const size_t dbytes = tab.size() * sizeof(double), ibytes = (nxs.size() + offs.size()) * sizeof(int32_t);
  CK(cudaSetDevice(h->device));
  void* dev = nullptr;
  CK(cudaMalloc(&dev, dbytes + ibytes));
  cudaError_t e = cudaMemcpy(dev, tab.data(), dbytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy((char*)dev + dbytes, nxs.data(), nxs.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (e == cudaSuccess)
    e = cudaMemcpy((char*)dev + dbytes + nxs.size() * sizeof(int32_t), offs.data(), offs.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { cudaFree(dev); return fail(FOT_ERR_CUDA, "fot_add_route: upload", e); }
  if (h->routes_dev) cudaFree(h->routes_dev);
  h->routes_dev = dev;
  h->rt_tab.swap(tab); h->rt_nx.swap(nxs); h->rt_off.swap(offs);
  h->max_nx = std::max(h->max_nx, nx);
  *route_id = h->rt_nx[0] - 1;
  return FOT_OK;
}

extern "C" int fot_set_routes(fot_handle_t* h, const int32_t* route) {
  if (!h) return fail(FOT_ERR_ARG, "fot_set_routes: null handle");
  h->route_ids = route;
  return FOT_OK;
}

extern "C" int fot_peer_alloc(int device, size_t bytes, void** ptr, unsigned char handle[64]) {
  if (!ptr || !handle || bytes == 0) return fail(FOT_ERR_ARG, "fot_peer_alloc: bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  CK(cudaSetDevice(device));
  CK(cudaMalloc(ptr, bytes));
  CK(cudaMemset(*ptr, 0, bytes));
  cudaIpcMemHandle_t hd;
  cudaError_t e = cudaIpcGetMemHandle(&hd, *ptr);
  if (e != cudaSuccess) { cudaFree(*ptr); *ptr = nullptr; return fail(FOT_ERR_CUDA, "cudaIpcGetMemHandle", e); }
  memcpy(handle, &hd, 64);
  return FOT_OK;
}

extern "C" int fot_peer_open(int device, const unsigned char handle[64], void** ptr) {
  if (!ptr || !handle) return fail(FOT_ERR_ARG, "fot_peer_open: bad argument");
  CK(cudaSetDevice(device));
  cudaIpcMemHandle_t hd;
  memcpy(&hd, handle, 64);
  CK(cudaIpcOpenMemHandle(ptr, hd, cudaIpcMemLazyEnablePeerAccess));
  return FOT_OK;
}

extern "C" int fot_peer_close(void* ptr) {
  if (ptr) CK(cudaIpcCloseMemHandle(ptr));
  return FOT_OK;
}

extern "C" int fot_peer_free(void* ptr) {
  if (ptr) CK(cudaFree(ptr));
  return FOT_OK;
}

extern "C" int fot_peer_await(int device, void* stream, const void* flags, int world, unsigned seq, void* err_word) {
  if (!flags || !err_word || world < 1 || world > 1024) return fail(FOT_ERR_ARG, "fot_peer_await: bad argument");
  CK(cudaSetDevice(device));
  fot_await_kernel<<<1, (world + 31) / 32 * 32, 0, (cudaStream_t)stream>>>((const unsigned*)flags, world, seq, 2000000000ll, (unsigned*)err_word);
  CK(cudaGetLastError());
  return FOT_OK;
}

extern "C" int fot_fetch_winners(fot_handle_t* h, int q0, int n, double* out) {
  if (!h || !out || q0 < 0 || n < 1) return fail(FOT_ERR_ARG, "fot_fetch_winners: bad argument");
  if (!h->last_winner_d || q0 + n > h->last_winner_nq) return fail(FOT_ERR_ARG, "fot_fetch_winners: no such queries in the last host-result call");
  CK(cudaSetDevice(h->device));
  const size_t row = (size_t)FOT_N_SERIES * h->plan.n_t_max;
  CK(cudaMemcpyAsync(out, h->last_winner_d + (size_t)q0 * row, (size_t)n * row * sizeof(double), cudaMemcpyDeviceToHost, h->d2h_stream));
  CK(cudaStreamSynchronize(h->d2h_stream));
  return FOT_OK;
}

extern "C" float fot_last_kernel_ms(const fot_handle_t* h) {
  if (!h || !h->timed) return -1.0f;
  float ms = -1.0f;
  if (cudaEventSynchronize(h->ev1) != cudaSuccess) return -1.0f;
  if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) != cudaSuccess) return -1.0f;
  return ms;
}

extern "C" int fot_last_sweep_kind(const fot_handle_t* h) { return h ? h->last_sweep_kind : 0; }
extern "C" int fot_last_pair_features(const fot_handle_t* h) { return h && h->last_sweep_kind == 4 ? h->last_pair_feat : -1; }

extern "C" int fot_launch_stage_ms(const fot_handle_t* h, int back, float ms[3]) {
  if (!h || !ms || back < 0 || back >= fot_handle::kRing || back >= h->n_launch)
    return fail(FOT_ERR_ARG, "fot_launch_stage_ms: no such launch");
  const cudaEvent_t* ring = h->ring.data() + (size_t)((h->n_launch - 1 - back) % fot_handle::kRing) * 4;
  CK(cudaEventSynchronize(ring[3]));
  for (int i = 0; i < 3; ++i) CK(cudaEventElapsedTime(&ms[i], ring[i], ring[i + 1]));
  return FOT_OK;
}

extern "C" int fot_probe_fma_tflops(int device, int kind, double* tflops_out) {
  if (!tflops_out || kind < 0 || kind > 2) return fail(FOT_ERR_ARG, "fot_probe_fma_tflops: bad argument");
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return fail(FOT_ERR_NO_DEVICE, "no CUDA device");
  CK(cudaSetDevice(device));
  int sms = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  float* sink = nullptr;
  CK(cudaMalloc(&sink, 4));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  const int blocks = sms * 8, threads = 256, iters = kind == 0 ? 4096 : 8192;
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    CK(cudaEventRecord(e0));
    if (kind == 0) fot_probe_kernel<0><<<blocks, threads>>>(sink, iters);
    else if (kind == 1) fot_probe_kernel<1><<<blocks, threads>>>(sink, iters);
    else fot_probe_kernel<2><<<blocks, threads>>>(sink, iters);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    const double fmas = (double)blocks * threads * iters * 64.0 * (kind == 2 ? 2.0 : 1.0);
    const double tf = 2.0 * fmas / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(sink);
  CK(cudaGetLastError());
  *tflops_out = best;
  return FOT_OK;
}

// ---- prediction post-processing (SURVEY.md section 8f, rank 1) ------------------------------------------
static int pred_begin(int device, const char* what) {
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return fail(FOT_ERR_NO_DEVICE, "no CUDA device (this library has no CPU path)");
  if (device < 0 || device >= n_dev) return fail(FOT_ERR_ARG, what);
  CK(cudaSetDevice(device));
  return FOT_OK;
}
static int pred_end(void* stream) {
  CK(cudaGetLastError());
  if (!stream) CK(cudaStreamSynchronize(nullptr));
  return FOT_OK;
}

extern "C" int fot_predict_cv_device(int device, void* stream, int n_q, int P, const double* p_curr, const double* p_prev,
                                     const double* staleness, double sgan_dt, const double* time_target, int n_steps,
                                     const double* cur_pos, int obs_float32, double* out) {
  if (n_q < 1 || P < 1 || n_steps < 1 || !p_curr || !time_target || !out || !(sgan_dt > 0.0))
    return fail(FOT_ERR_ARG, "fot_predict_cv_device: bad argument");
  int rc = pred_begin(device, "fot_predict_cv_device: bad device ordinal");
  if (rc != FOT_OK) return rc;
  const int T_out = n_steps + (cur_pos ? 1 : 0);
  const size_t smem = (size_t)P * 2 * sizeof(double);
  if (smem > 48 * 1024) return fail(FOT_ERR_TOO_LARGE, "fot_predict_cv_device: too many pedestrians per query");
  // the kernel's static shared memory comes on top: near 48 KB of dynamic shared memory the launch needs the opt-in
  if (smem > 32 * 1024) CK(cudaFuncSetAttribute(fot_cv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  fot_cv_kernel<<<n_q, 256, smem, (cudaStream_t)stream>>>(p_curr, p_prev, staleness, time_target, cur_pos, out, P, n_steps,
                                                          T_out, sgan_dt, obs_float32);
  return pred_end(stream);
}

extern "C" int fot_process_prediction_device(int device, void* stream, int n_q, int S, int P, int pred_len, const double* pred,
                                             const double* anchor, const double* staleness, double sgan_dt,
                                             const double* time_target, int n_steps, double* out) {
  if (n_q < 1 || S < 1 || P < 1 || pred_len < 1 || pred_len > kPredLenMax || n_steps < 1 || !pred || !time_target || !out ||
      !(sgan_dt > 0.0))
    return fail(FOT_ERR_ARG, "fot_process_prediction_device: bad argument (pred_len <= 64)");
  int rc = pred_begin(device, "fot_process_prediction_device: bad device ordinal");
  if (rc != FOT_OK) return rc;
  const int threads = std::min(256, std::max(32, (2 * P + 31) / 32 * 32));
  fot_resample_kernel<<<(unsigned)((long long)n_q * S), threads, 0, (cudaStream_t)stream>>>(pred, anchor, staleness, time_target, out, S, P,
                                                                                            pred_len, n_steps, sgan_dt);
  return pred_end(stream);
}

extern "C" int fot_select_best_sample_device(int device, void* stream, int n_q, int S, int P, int T, const double* samples,
                                             double* dist_scratch, int32_t* best_idx) {
  if (n_q < 1 || S < 1 || P < 1 || T < 1 || !samples || !dist_scratch || !best_idx)
    return fail(FOT_ERR_ARG, "fot_select_best_sample_device: bad argument");
  int rc = pred_begin(device, "fot_select_best_sample_device: bad device ordinal");
  if (rc != FOT_OK) return rc;
  const long long n = (long long)n_q * S;
  fot_best_dist_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(samples, dist_scratch, n_q, S, P * T);
  fot_best_pick_kernel<<<(n_q + 127) / 128, 128, 0, (cudaStream_t)stream>>>(dist_scratch, best_idx, n_q, S);
  return pred_end(stream);
}

extern "C" int fot_prepend_current_device(int device, void* stream, int n_q, int S, int P, int T, const double* in,
                                          const int32_t* pick, const double* cur_pos, int conditional, double* out) {
  if (n_q < 1 || S < 1 || P < 1 || T < 1 || !in || !cur_pos || !out)
    return fail(FOT_ERR_ARG, "fot_prepend_current_device: bad argument");
  int rc = pred_begin(device, "fot_prepend_current_device: bad device ordinal");
  if (rc != FOT_OK) return rc;
  const long long blocks = (long long)n_q * (pick ? 1 : S);
  fot_prepend_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(in, pick, cur_pos, out, S, P, T, conditional);
  return pred_end(stream);
}

extern "C" int fot_safety_metrics_device(int device, void* stream, int n_q, int P, const double* ego, const double* ped_pos,
                                         const double* ped_vel, const int32_t* n_peds, double combined_radius,
                                         const double* offsets, int n_circ, double* out) {
  if (n_q < 1 || P < 0 || !ego || !out || (P > 0 && (!ped_pos || !ped_vel)) || n_circ < 0 || n_circ > FOT_MAX_CIRCLES ||
      (n_circ > 0 && !offsets))
    return fail(FOT_ERR_ARG, "fot_safety_metrics_device: bad argument");
  int rc = pred_begin(device, "fot_safety_metrics_device: bad device ordinal");
  if (rc != FOT_OK) return rc;
  CircleOffsets off{};
  for (int i = 0; i < n_circ; ++i) off.v[i] = offsets[i];
  const long long threads = (long long)n_q * 32;
  fot_safety_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ego, ped_pos, ped_vel, n_peds, out, n_q, P,
                                                                                         combined_radius, off, n_circ);
  return pred_end(stream);
}

// ---- nearest point on the reference path (DESIGN.md section 4e) -----------------------------------------
extern "C" int fot_nearest_s_device(fot_handle_t* h, void* stream, int n, const double* x, const double* y,
                                    const double* prev_s, double* s_out, int32_t* status) {
  if (!h || n < 0 || (n > 0 && (!x || !y || !prev_s || !s_out || !status)))
    return fail(FOT_ERR_ARG, "fot_nearest_s_device: bad argument");
  if (n == 0) return FOT_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  if (!stream) {                 // the handle's stream does not synchronise with the legacy default stream on its own:
    CK(cudaEventRecord(h->ev_join, cudaStreamLegacy));   // inputs written there (plain or pinned async copies) come first
    CK(cudaStreamWaitEvent(st, h->ev_join, 0));
  }
  const int threads = 256, per_block = threads / 32;
  const unsigned blocks = (unsigned)((n + per_block - 1) / per_block);
  if (h->route_ids) fot_nearest_s_routed<<<blocks, threads, 0, st>>>(h->plan, routes_of(h, 0), n, x, y, prev_s, s_out, status);
  else fot_nearest_s<<<blocks, threads, 0, st>>>(h->plan, n, x, y, prev_s, s_out, status);
  CK(cudaGetLastError());
  if (!stream) CK(cudaStreamSynchronize(st));
  return FOT_OK;
}

#ifdef FOT_PHASE_CLOCKS
// tuning aid: read and reset the per-phase clock accumulators of fot_sweep_items
extern "C" int fot_debug_phase_clocks(unsigned long long out[16]) {
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpyFromSymbol(out, fot::g_phase_clk, sizeof(unsigned long long) * 16));
  unsigned long long z[16] = {};
  CK(cudaMemcpyToSymbol(fot::g_phase_clk, z, sizeof z));
  return FOT_OK;
}
#endif
