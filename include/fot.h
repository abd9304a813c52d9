/*
 * fot.h -- C ABI of the B200-native Frenet optimal-trajectory candidate sweep.
 *
 * This is the drop-in boundary for ONE hot path of mnhrk15/integrated_path_planning:
 * everything `FrenetPlanner.plan()` does between "ego state already in the Frenet
 * frame" and "best FrenetPath selected"  (reference src/planning/frenet_planner.py:271-294,
 * i.e. _generate_frenet_paths :376, _generate_brake_candidates :453, _calc_global_paths :736,
 * _check_paths :891, _apply_stop_distance_filter :307, _select_best_path :1235).
 * The reference has no FFI of its own (it is pure Python); these entry points are what a
 * ctypes binding of that path binds.  Plain pointers and sizes only -- no torch types.
 *
 * Conventions
 *   - all floating point is IEEE binary64 ("double"), as in the reference;
 *   - "device" pointers are CUDA device pointers on the handle's device (e.g. torch
 *     tensor .data_ptr()); "host" pointers are ordinary process memory;
 *   - every function returns FOT_OK (0) or a negative FOT_ERR_* code; "no valid path"
 *     is NOT an error: best_idx = -1 (reference returns None, frenet_planner.py:298-299).
 *   - candidate index = generation order of the reference (:398-449):
 *     ((j_T * n_v + k_v) * n_d + i_d), brake-ladder candidates appended after the grid.
 */
#ifndef FOT_H_
#define FOT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FOT_ABI_VERSION 8   /* 2: + prediction post-processing and safety metrics; 3: + fot_plan_batch_device_to_host;
                               4: + fot_result_t.winner_samples, fot_fetch_winners, fot_reload_options;
                               5: + fot_set_result_mirror, fot_peer_* (gather of a sharded sweep over peer memory);
                               6: + fot_last_sweep_kind, fot_last_pair_features (fot_sweep_pairs is the default sweep kernel);
                               7: + fot_nearest_s_device (nearest point on the path, certified against the host);
                               8: + fot_ranked_t, fot_rank_candidates (the k best feasible candidates per query) */
#define FOT_ABI_MINOR 1     /* additions within a version that change no existing struct, entry point or behaviour, so a
                               caller built against an earlier minor of the same version keeps working; 0 at each new
                               version.  Version 8: 1: + fot_weighted_t, fot_select_weighted, fot_cost_terms (winners
                               under many cost weightings, the five cost terms per candidate); + fot_route_t,
                               fot_add_route, fot_set_routes (every query on its own reference path); then, still under
                               minor 1, + fot_assessed_t, fot_assess_trajectories, then fot_assess_candidates:
                               fot_abi_minor() does not tell whether a library has them, a caller looks the symbol up
                               (DESIGN.md sections 4i, 4j) */
#define FOT_MAX_CIRCLES 8
#define FOT_MAX_RANKED 32
#define FOT_N_STATS 8    /* ok, max_speed, max_accel, max_curvature, max_lat_accel, road_bound, collision, stop_distance */
#define FOT_N_SERIES 15  /* t s s_d s_dd s_ddd d d_d d_dd d_ddd x y yaw c v a  (data_structures.py:149-181) */

/* candidate categories (frenet_planner.py:910-918, :324; DROP = silently discarded :933-956) */
enum {
  FOT_CAT_OK = 0, FOT_CAT_SPEED = 1, FOT_CAT_ACCEL = 2, FOT_CAT_CURV = 3, FOT_CAT_LAT = 4,
  FOT_CAT_ROAD = 5, FOT_CAT_COLL = 6, FOT_CAT_STOP = 7, FOT_CAT_DROP = 8
};

enum {
  FOT_OK = 0,
  FOT_ERR_ARG = -1,        /* bad argument / unsupported size */
  FOT_ERR_CUDA = -2,       /* CUDA runtime error (see fot_last_error) */
  FOT_ERR_NO_DEVICE = -3,  /* no CUDA device: there is no CPU fallback */
  FOT_ERR_TOO_LARGE = -4   /* batch shape beyond the sweep: time grid over 320 samples, lateral grid over 8192 targets,
                              S*P or static points over 32768, tables beyond shared memory (fot_last_error names it) */
};

/* dynamic-obstacle modes (frenet_planner.py:1043-1047) */
enum { FOT_DYN_NONE = 0, FOT_DYN_SINGLE = 1, FOT_DYN_DISTRIBUTION = 2 };

/* Planner-constant knobs: FrenetPlanner.__init__ (frenet_planner.py:149-210). */
typedef struct fot_config {
  double dt;               /* :171 */
  double max_speed;        /* constructor value; teleport guard uses max(override, this) (:955) */
  double max_road_width;   /* road-bound check (:982) */
  double k_j, k_t, k_d, k_s_dot, k_lat, k_lon;   /* :187-192 */
  double collide_r2;       /* sq_rubicon     = max(ego_radius + obstacle_radius, 1e-6) ** 2            (:1172-1174) */
  double collide_r2_single;/* sq_rubicon_dyn = (that radius * collision_margin_inflation) ** 2; used by the
                              single-sample dynamic test only (:1173-1175, :1072).  Both are evaluated by the
                              host with the reference's own expression so the thresholds are bit-identical. */
  double chance_epsilon;   /* :197 */
  double circle_offsets[FOT_MAX_CIRCLES]; /* EgoFootprint.offsets (footprint.py:66-81) */
  int32_t n_circles;       /* 0 = single circle at the path point (footprint None, :1152) */
  int32_t n_T;             /* horizon grid size (:397-398) */
  int32_t n_d;             /* lateral grid size (:419-420) */
  int32_t n_B;             /* brake-ladder horizons that fit max_t (:475-485) */
  int32_t n_total;         /* brake-candidate samples: round(max_t/dt)+1 (:473) */
  int32_t nx;              /* spline knots */
} fot_config_t;

/* Planner-constant tables, all HOST pointers (copied at create).
 * The horizon tables are built by the host exactly as the reference builds its TimeCache
 * (:586-617): n_steps = int(round(T/dt)); inv4/inv5 = numpy.linalg.inv of the quartic/quintic
 * boundary matrices (row-major 2x2 / 3x3).  The kernel applies them in the same accumulation
 * order as the reference's `b @ A_inv.T` (:640, :683). */
typedef struct fot_tables {
  const double*  T;        /* [n_T]   T_j = min_t + j*dt */
  const int32_t* n_steps;  /* [n_T]   */
  const double*  inv4;     /* [n_T][4] */
  const double*  inv5;     /* [n_T][9] */
  const double*  Tb;       /* [n_B]   brake horizons */
  const int32_t* n_steps_b;/* [n_B]   */
  const double*  inv4b;    /* [n_B][4] */
  const double*  inv5b;    /* [n_B][9] */
  const double*  d_grid;   /* [n_d]   lateral targets (:420) */
  /* natural cubic spline, CubicSpline1D coefficients (cubic_spline.py:23-45) */
  const double*  knots;    /* [nx] */
  const double*  xa; const double* xb; const double* xc; const double* xd; /* [nx],[nx-1],[nx],[nx-1] */
  const double*  ya; const double* yb; const double* yc; const double* yd;
} fot_tables_t;

/* One batch of independent planning queries (one reference plan() call each). */
typedef struct fot_batch {
  int32_t n_q;
  int32_t n_v_max;            /* row stride of v_grid */
  const double*  frenet;      /* [n_q][6]  s, s_d, s_dd, d, d_d, d_dd   (:371) */
  const double*  target_speed;/* [n_q]     (:232) */
  const double*  limits;      /* [n_q][4]  max_speed, max_accel, max_curvature, max_lat_accel after overrides (:921-930) */
  const double*  stop_dist;   /* [n_q]     max_stop_distance, NaN = None (:285) */
  const double*  v_grid;      /* [n_q][n_v_max] terminal-speed grid (:410-413) */
  const int32_t* n_v;         /* [n_q]     entries used in each v_grid row */
  const double*  static_obs;  /* [n_q or 1][n_static][2]  (:1181-1198); may be NULL when n_static == 0 */
  int32_t n_static;
  int32_t static_per_query;   /* 0: one set shared by all queries */
  const double*  dyn;         /* [n_q][S][P][T_obs][2] reference layout (:242, :246); NULL when dyn_mode == NONE */
  int32_t S, P, T_obs;
  int32_t dyn_mode;           /* FOT_DYN_* */
} fot_batch_t;

/* Results.  cand_cat / cand_cost are optional diagnostics (may be NULL). */
typedef struct fot_result {
  int32_t* best_idx;    /* [n_q]  generation-order index of the winner, -1 = none */
  double*  best_cost;   /* [n_q]  +inf when none */
  int32_t* stats;       /* [n_q][FOT_N_STATS]  last_check_stats counts (:291) */
  int32_t* winner_len;  /* [n_q]  samples kept after NaN-prefix truncation (:866) */
  double*  winner;      /* [n_q][FOT_N_SERIES][n_t_max]  winner sequences */
  uint8_t* cand_cat;    /* [n_q][cand_stride] or NULL */
  double*  cand_cost;   /* [n_q][cand_stride] or NULL */
  int32_t  cand_stride;
  int32_t  winner_samples; /* host-result entry points only: 0 = every series in full (row length n_t_max); k > 0 = only the
                              first min(k, n_t_max) samples of each series are copied back and `winner` is
                              [n_q][FOT_N_SERIES][k].  A closed-loop caller consumes sample 1 of the winner and nothing
                              else (integrated_simulator.py:660-667: get_state_at_index(1), c[1]); k = 2 cuts the
                              read-back from 6.1 KB to 240 B per query.  The full series of the last call stay on the
                              device: fot_fetch_winners.  Must be 0 for fot_plan_batch_device. */
} fot_result_t;

/* A handle owns one device's planner tables, streams and scratch buffers.  ONE fot_plan_batch_* call may be in flight per
 * handle: the calls share the handle's scratch (arg-min partials, cost tables, trajectory boxes) and timing events, so
 * launches on one handle must be stream-ordered with each other -- an asynchronous fot_plan_batch_device launch has to
 * be followed on the same stream, or synchronised, before the next call on that handle.  Use one handle per concurrent
 * caller (handles are cheap: < 1 MB plus scratch that grows with the batch). */
typedef struct fot_handle fot_handle_t;

/* ABI version of the loaded library, and its minor revision within that version (FOT_ABI_MINOR). */
int fot_abi_version(void);
int fot_abi_minor(void);
/* Human-readable text of the last error on this thread. */
const char* fot_last_error(void);

/* Replaces FrenetPlanner.__init__ for the sweep (frenet_planner.py:149-225): copies knobs,
 * horizon tables and spline coefficients to `device`, creates the stream and scratch. */
int fot_create(const fot_config_t* cfg, const fot_tables_t* tables, int device, fot_handle_t** out);
int fot_destroy(fot_handle_t* h);

/* Longest candidate (samples); the row length of fot_result_t.winner. */
int fot_n_t_max(const fot_handle_t* h);
/* Candidates of a query with n_v terminal speeds; brake ladder counted when has_brake != 0. */
int fot_candidate_count(const fot_handle_t* h, int n_v, int has_brake);

/* Replaces frenet_planner.py:271-294 for n_q queries.  All pointers in `batch` and `res` are
 * DEVICE pointers.  Asynchronous on `stream` (a cudaStream_t, NULL = the handle's own stream,
 * which is then synchronised before returning). */
int fot_plan_batch_device(fot_handle_t* h, const fot_batch_t* batch, const fot_result_t* res, void* stream);

/* ---- ranked alternatives (DESIGN.md section 4f) --------------------------------------------------------------------
 * For query q the ranked list holds the candidates the winner selection could pick, best first: category FOT_CAT_OK
 * after the stop-distance filter and a cost below +inf (a NaN cost never ranks, as it never wins), ordered by lower
 * cost first and, on exactly equal cost, lower generation index first -- the reference's tie rule (first strict
 * minimum, frenet_planner.py:1254-1257) extended to a ranking.  Rank 0 is therefore best_idx / best_cost of the same
 * launch.  Ranks past the last such candidate are padded: idx -1, cost +inf, len 0 (their series rows are not
 * written).  Series rows hold samples [0, N) of the candidate's N; the first len of them are what the reference keeps. */
typedef struct fot_ranked {
  int32_t  k;        /* 1 .. FOT_MAX_RANKED */
  int32_t* idx;      /* [n_q][k] generation-order index, -1 = no further feasible candidate */
  double*  cost;     /* [n_q][k] +inf where idx == -1 */
  int32_t* len;      /* [n_q][k] samples kept after NaN-prefix truncation, or NULL */
  double*  series;   /* [n_q][k][FOT_N_SERIES][n_t_max], or NULL (needs len) */
} fot_ranked_t;
/* The k best candidates of every query from the per-candidate table a fot_plan_batch_device launch of the same batch
   wrote (cand_cat / cand_cost / cand_stride), with their 15 series regenerated as fot_winner does.  DEVICE pointers;
   stream-ordered after that launch on `stream` (NULL: the handle's stream, synchronised). */
int fot_rank_candidates(fot_handle_t* h, const fot_batch_t* batch, const uint8_t* cand_cat, const double* cand_cost,
                        int cand_stride, const fot_ranked_t* out, void* stream);

/* ---- cost-weight sweeps (DESIGN.md section 4g) ---------------------------------------------------------------------
 * No cost weight affects a candidate's category; the weights enter only the cost, a fixed expression of five
 * per-candidate terms (frenet_planner.py:703-734):
 *   lat = k_j*Jp + k_t*Jt + k_d*Jd      Jp = sum d'''^2, Jd = d_end^2
 *   lon = k_j*Js + k_t*Jt + k_s_dot*Jv  Js = sum s'''^2, Jv = (target_speed - s_d[-1])^2, Jt = t[-1]
 *   cost_w = k_lat*lat + k_lon*lon
 * evaluated left to right, every product and sum rounded on its own (no contraction).  For query q and weighting
 * w = (k_j, k_t, k_d, k_s_dot, k_lat, k_lon) the selected candidate is the one a planner created with w returns for the
 * same inputs: among the candidates whose table category is FOT_CAT_OK, the smallest cost_w below +inf, and on exactly
 * equal cost the lower generation index (first strict minimum, frenet_planner.py:1254-1257).  A NaN or infinite cost_w
 * never wins, so a NaN weight gives no winner.  No winner: idx -1, cost +inf, len 0, series row not written.  For w
 * equal to the handle's own weights the selection is best_idx / best_cost / winner of the same launch. */
#define FOT_MAX_WEIGHT_SETS 256
typedef struct fot_weighted {
  int32_t n_w;              /* 1 .. FOT_MAX_WEIGHT_SETS */
  int32_t per_query;        /* 0: one list of n_w weightings for every query; 1: a list per query */
  const double* weights;    /* [(n_q | 1)][n_w][6]  k_j k_t k_d k_s_dot k_lat k_lon */
  int32_t* idx;             /* [n_q][n_w]  generation-order index, -1 = no candidate */
  double*  cost;            /* [n_q][n_w]  +inf where idx == -1 */
  int32_t* len;             /* [n_q][n_w] samples kept after NaN-prefix truncation, or NULL */
  double*  series;          /* [n_q][n_w][FOT_N_SERIES][n_t_max], or NULL (needs len) */
} fot_weighted_t;
/* The winner of every query under each of n_w weightings, from the per-candidate table (cand_cat, cand_stride) a
   fot_plan_batch_device launch of the same batch wrote, with the winners' series regenerated as fot_winner does.
   DEVICE pointers; stream-ordered after that launch on `stream` (NULL: the handle's stream, synchronised). */
int fot_select_weighted(fot_handle_t* h, const fot_batch_t* batch, const uint8_t* cand_cat, int cand_stride,
                        const fot_weighted_t* out, void* stream);
/* The five cost terms of every generated candidate, for cost learning: terms[n_q][cand_stride][5] = (Jp, Jd, Js, Jv, Jt)
   as above, NaN past the query's candidates (fot_candidate_count).  Every candidate has its terms whatever its category
   (the reference computes the cost before the checks).  Needs only the batch's frenet, target_speed, v_grid and n_v;
   no sweep.  DEVICE pointers; asynchronous on `stream` (NULL: the handle's stream, synchronised). */
int fot_cost_terms(fot_handle_t* h, const fot_batch_t* batch, int cand_stride, double* terms, void* stream);

/* DEVICE inputs (`batch`), HOST results (`res`): for a caller whose obstacle tensor is produced on the GPU (the
 * entry points below) and whose winners are consumed on the host -- frenet_planner.py:271-294 for n_q queries
 * behind integrated_simulator.py:447-525.  Queries are swept in ranges and each range's winners are copied back
 * while the next range runs.  `stream`: the cudaStream_t on which the inputs become ready (NULL: ready now).
 * Returns when the results are in `res` (page-locked result arrays make the copies asynchronous). */
int fot_plan_batch_device_to_host(fot_handle_t* h, const fot_batch_t* batch, const fot_result_t* res, void* stream);

/* Same call with HOST pointers everywhere: stages the small per-query arrays through the handle's
 * pinned buffers, uploads the obstacle tensor straight from the caller's memory, runs the kernels,
 * copies the results back, and returns when they are in `res`. This is the entry point
 * FrenetPlanner.plan() binds.  Large batches are pipelined: the tensor goes up in slices while the
 * sweep is already running (every CTA waits for the slice of its own query), and the winners of the
 * first queries come back while the last are still swept.  Page-locked (pinned) `batch->dyn` and
 * result arrays make those copies true asynchronous DMAs; pageable memory works but serialises. */
int fot_plan_batch_host(fot_handle_t* h, const fot_batch_t* batch, const fot_result_t* res);

/* ---- multi-GPU: the one gather of a query-sharded sweep (SURVEY.md section 8e), without a collective call -----------
 * Queries shard over GPUs with no traffic during compute; the winners (6.2 KB per query) have to reach one place.
 * fot_set_result_mirror gives a handle a SECOND destination for the winner block of every following
 * fot_plan_batch_device launch: five DEVICE pointers laid out like fot_result_t's (best_idx, best_cost, stats,
 * winner_len, winner; cand_* ignored), typically a slice of a buffer on the gather root mapped into this process over
 * NVLink peer memory (fot_peer_open).  The winner kernel stores every value twice, locally and into the mirror, so the
 * block is on the root when the launch completes; `flag` (device pointer, may be peer memory, or NULL) receives the
 * number of mirrored launches since this flag word was set -- 1, 2, 3, ... -- behind each of them (a system-scope fence
 * precedes the write).
 * mirror = NULL switches it off. */
int fot_set_result_mirror(fot_handle_t* h, const fot_result_t* mirror, void* flag);
/* Peer-memory plumbing (CUDA IPC; one process per GPU): the root allocates a buffer with fot_peer_alloc and hands the
 * 64-byte handle to the other ranks (any byte transport), which map it with fot_peer_open.  The buffer is zeroed. */
int fot_peer_alloc(int device, size_t bytes, void** ptr, unsigned char handle[64]);
int fot_peer_open(int device, const unsigned char handle[64], void** ptr);
int fot_peer_close(void* ptr);
int fot_peer_free(void* ptr);
/* Root side: enqueue on `stream` a wait until flags[0 .. world) have all reached sequence number `seq` (what the
 * ranks' mirrored launches publish); gives up after 2 s and sets *err_word (device pointer, 4 bytes) to 1. */
int fot_peer_await(int device, void* stream, const void* flags, int world, unsigned seq, void* err_word);

/* Full winner series of queries [q0, q0 + n) of the LAST fot_plan_batch_host / _device_to_host call on this handle,
 * from the device-resident result block into out[n][FOT_N_SERIES][n_t_max] (HOST pointer).  For callers that asked for
 * winner_samples > 0 and need the whole trajectory of a few queries after all (logging, plotting). */
int fot_fetch_winners(fot_handle_t* h, int q0, int n, double* out);

/* The FOT_* tuning environment variables (chunking / gating of the host-pointer call, kernel choice, queue capacity;
 * listed in csrc/fot_api.cu `struct Options`) are resolved ONCE, in fot_create; no planning call reads the environment.
 * This re-reads them for handle `h` (NULL: every live handle of the process): the tests and tuning scripts switch
 * variants on a live handle with it. */
int fot_reload_options(fot_handle_t* h);

/* Device-side time of the kernels of the last fot_plan_batch_* call on this handle, in ms (CUDA events; for a call that
 * was cut into chunks / ranges: from the first chunk's start to the last kernel of any chunk); negative if unavailable. */
float fot_last_kernel_ms(const fot_handle_t* h);

/* Which sweep kernel the last launch on this handle used: 4 fot_sweep_pairs (one longitudinal profile per warp; the
 * default), 1 fot_sweep_items (sample-major with block barriers; shapes beyond the limits of fot_sweep_pairs), 0 none
 * yet; 2 (the retired candidate-major kernel) is never returned. */
int fot_last_sweep_kind(const fot_handle_t* h);

/* fot_sweep_pairs is compiled per set of optional modes (1 static obstacles, 2 footprint circles, 4 violation budget,
 * 8 per-candidate outputs, 16 unstaged obstacle block / unsorted lateral grid, 32 per-query routes; DESIGN.md sections
 * 4d, 4h) and the smallest instantiated superset of what a batch needs runs: the set of the last launch, or -1 if
 * another kernel ran. */
int fot_last_pair_features(const fot_handle_t* h);

/* Device time of the three stages of the `back`-th most recent launch on this handle (0 = the
 * last one; the handle keeps the last 256), in ms, from CUDA events on the launching stream:
 * ms[0] obstacle prepass, ms[1] sweep kernel, ms[2] winner kernel.  Waits for that launch. */
int fot_launch_stage_ms(const fot_handle_t* h, int back, float ms[3]);

/* Pipe-throughput probes used to anchor the roofline denominator (MEASURED_PEAKS.json holds no
 * FP64/FP32 figure).  kind: 0 = FP64 FMA, 1 = FP32 FMA, 2 = packed FP32x2 FMA.
 * Writes achieved TFLOP/s (2 flops per FMA). */
int fot_probe_fma_tflops(int device, int kind, double* tflops_out);

/* ---- routes: every query on its own reference path (DESIGN.md section 4h) ------------------------------------------
 * A handle plans on the path given to fot_create (route 0) and on any number of further paths registered with
 * fot_add_route.  Only the path is per query: grids, dt, radii, cost weights and footprint stay the handle's.  A query
 * on route r gives, bit for bit, what a handle created with route r's path gives for it. */
typedef struct fot_route {   /* one more reference path: CubicSpline1D coefficients as in fot_tables_t, HOST pointers */
  int32_t nx;                /* >= 2 knots */
  const double* knots;       /* [nx] */
  const double *xa, *xb, *xc, *xd, *ya, *yb, *yc, *yd;   /* [nx], [nx-1], [nx], [nx-1] */
} fot_route_t;
/* Copies a path to the handle's device; *route_id = 1, 2, ...  Route 0 is the path of fot_create.
   Not while a call on this handle is in flight (it may reallocate the route tables). */
int fot_add_route(fot_handle_t* h, const fot_route_t* route, int32_t* route_id);
/* DEVICE pointer: route[i] is the route of query i (point i) of every following fot_plan_batch_device,
   fot_plan_batch_device_to_host, fot_plan_batch_host, fot_rank_candidates, fot_select_weighted and
   fot_nearest_s_device call on this handle; the array must cover that call's n_q (n) and stay valid until the call
   has finished.  It is device memory for fot_plan_batch_host too.  NULL: every query on route 0, i.e. the behaviour
   without routes.  A route id outside [0, n_routes) plans nothing for that query (best_idx -1, best_cost +inf, stats
   zero, no ranked or weighted entry, its cand_cat entries left unwritten; the search gives s_out NaN, status 1) and no
   route table is read for it.
   Kernel choice and shared memory of a launch with a binding follow the LONGEST registered route: fot_sweep_pairs when
   it has at most 48 knots, else fot_sweep_items, which keeps the tables in shared memory up to 128 knots. */
int fot_set_routes(fot_handle_t* h, const int32_t* route);

/* ---- trajectory assessment (DESIGN.md section 4i) -------------------------------------------------------------------
 * How close m trajectories per query come to an obstacle field, and how many of its samples they collide with, in the
 * reference's collision geometry (collision_geometry / hits_static / hits_dynamic, frenet_planner.py:1126-1233).  The
 * trajectories are series blocks [n_q][m][FOT_N_SERIES][n_t] -- the layout of fot_result_t.winner, fot_ranked_t.series
 * and fot_weighted_t.series, with n_t = fot_n_t_max -- of which samples [0, len[q][j]) of rows t, x, y and yaw are read
 * (len is clipped to [0, n_t]).  The field is the dyn / S / P / T_obs / static_obs / n_static / static_per_query part of
 * a fot_batch_t of the same n_q queries (dyn_mode FOT_DYN_NONE: no dynamic obstacles; any S is accepted).
 *   circle centres  (x, y), or (x, y) + offset * (cos yaw, sin yaw) for each footprint circle of the handle
 *   time index      k = clip(rint(t / dt), 0, T_obs - 1) with the handle's dt (a NaN t gives 0)
 *   distance        d2 = dx*dx + dy*dy, unfused; a NaN d2 is neither a minimum nor a hit
 *   NaN rule        a pedestrian trajectory with a NaN at any step is ignored entirely (the reference's box prefilter)
 * Outputs per (q, j), for the n_r threshold pairs r2[i] = (r2_dyn, r2_static) of squared centre distances:
 *   dyn_min    [n_q][m]       sqrt of the smallest d2 to any dynamic obstacle sample, +inf if there is none
 *   dyn_at     [n_q][m][4]    (n, circle, s, p) of that minimum; ties go to the first entry in C order of an
 *                             [len, n_circ, S, P] array (np.argmin); -1 if there is none
 *   static_min [n_q][m], static_at [n_q][m][3]   the same for the static points, in order (n, circle, point)
 *   dyn_hits   [n_q][m][n_r]  obstacle samples s in [0, S) where some sample, circle and pedestrian has d2 <= r2_dyn
 *   first_hit  [n_q][m][n_r]  first trajectory sample n with a dynamic (d2 <= r2_dyn) or static (d2 <= r2_static) hit, -1
 *   static_hit [n_q][m][n_r]  1 if some static point lies within r2_static, else 0
 * With the handle's own pair -- (collide_r2_single, collide_r2) for a single-sample field, (collide_r2, collide_r2) for a
 * distribution -- a trajectory is collision-free in the planner's sense iff static_hit == 0 and
 * dyn_hits <= floor(chance_epsilon * S) (dyn_hits == 0 for a single sample).  A slot with len 0 (padded ranks, queries
 * without a winner) gives +inf, -1 and 0.  Footprint centres use CUDA cos / sin: with circles, distances may differ
 * from NumPy's by a few ulp (DESIGN.md 4b, 4i); with the single centre circle they are bit-identical. */
#define FOT_MAX_ASSESSED 256   /* trajectories per query */
#define FOT_MAX_RADII 16       /* threshold pairs */
#define FOT_MAX_ASSESS_NT 320  /* series row length */
typedef struct fot_assessed {
  int32_t m;                /* 1 .. FOT_MAX_ASSESSED */
  int32_t n_t;              /* row length of the series block, 1 .. FOT_MAX_ASSESS_NT */
  int32_t n_r;              /* 1 .. FOT_MAX_RADII */
  const double*  series;    /* [n_q][m][FOT_N_SERIES][n_t] */
  const int32_t* len;       /* [n_q][m] samples to assess */
  const double*  r2;        /* [n_r][2] (r2_dyn, r2_static) */
  double*  dyn_min;         /* [n_q][m] */
  int32_t* dyn_at;          /* [n_q][m][4] */
  double*  static_min;      /* [n_q][m] */
  int32_t* static_at;       /* [n_q][m][3] */
  int32_t* dyn_hits;        /* [n_q][m][n_r] */
  int32_t* first_hit;       /* [n_q][m][n_r] */
  int32_t* static_hit;      /* [n_q][m][n_r] */
} fot_assessed_t;
/* Assess the trajectories of `a` against the field `obstacles` (its query arrays are not read).  DEVICE pointers;
   stream-ordered on `stream` behind the launch that wrote the series (NULL: the handle's stream, synchronised). */
int fot_assess_trajectories(fot_handle_t* h, const fot_batch_t* obstacles, const fot_assessed_t* a, void* stream);

/* ---- candidate assessment (DESIGN.md section 4j) --------------------------------------------------------------------
 * The assessment above for EVERY generated candidate of every query, including those the sweep rejects, without a
 * sweep and without writing a series anywhere: each candidate is regenerated on chip and reduced there.
 *   candidates  those query q generates, in generation order -- the grid, then the brake ladder when the query
 *               generates it (initial s_d > 0.1): the columns of cand_cat and fot_cost_terms.  Column i of
 *               [n_q][cand_stride] is candidate i; columns past the query's candidates (fot_candidate_count) are blank.
 *   samples     [0, keep) with keep the reference's kept length (fp.py:826-833, :866): N when no x is NaN, else the
 *               first NaN index when it is >= 2, else 0; a finite q = 1 - kappa_ref * d <= 0.05 at any sample makes x[0]
 *               NaN and so keep 0.  keep == 0 gives a blank column: +inf, -1 and 0.
 *   series      t, x, y and yaw of a candidate are the values fot_rank_candidates / fot_winner write for it, bit for bit
 *               (the same time table, profile, spline and Frenet-to-Cartesian functions, yaw = wrap_angle).
 * Everything else -- circle centres, time index, unfused d2, the NaN rule, the (d2, flat index) tie order, the threshold
 * pairs and the outputs -- is fot_assess_trajectories', so column i equals what fot_assess_trajectories returns for
 * candidate i's series with len = keep.  Under the handle's own pair a candidate of category FOT_CAT_OK, FOT_CAT_COLL or
 * FOT_CAT_STOP is collision-free iff its category is not FOT_CAT_COLL.  The query's route follows fot_set_routes; a route
 * id out of range gives blank columns and reads no route table.
 *   queries  frenet, target_speed, v_grid, n_v, n_v_max and n_q of a fot_batch_t (what fot_cost_terms reads)
 *   field    the dyn / S / P / T_obs / dyn_mode / static_obs / n_static / static_per_query part of a fot_batch_t of the
 *            same n_q queries, as for fot_assess_trajectories: the planning field or another one
 *   out      a fot_assessed_t with m == cand_stride (FOT_MAX_ASSESSED does not bound it here), series and len NULL,
 *            n_t ignored; its outputs are [n_q][cand_stride][...]
 *   keep     [n_q][cand_stride] kept samples per column (0 for blank columns), or NULL
 * DEVICE pointers; asynchronous on `stream` (NULL: the handle's stream, synchronised).  Declared under FOT_ABI_MINOR 1:
 * a caller looks the symbol up. */
int fot_assess_candidates(fot_handle_t* h, const fot_batch_t* queries, const fot_batch_t* field, int cand_stride,
                          const fot_assessed_t* out, int32_t* keep, void* stream);

/* ---- next row (SURVEY.md section 8f, rank 1): the predictor's post-processing on the device ---------
 * Builds the obstacle tensor fot_batch_t.dyn consumes, so that batched roll-outs never upload it.
 * All pointers are DEVICE pointers; `stream` is a cudaStream_t (NULL = the default stream, synchronised
 * before returning).  The time grid `time_target[n_steps]` is the reference's
 * np.arange(sim_dt, max(plan_horizon, pred_len * sgan_dt) + 1e-9, sim_dt) (trajectory_predictor.py:214-215,
 * :283-284), built by the caller with NumPy so that its values are bit-identical. */

/* Replaces TrajectoryPredictor.predict_cv (trajectory_predictor.py:188-231).
 *   p_curr, p_prev [n_q][P][2]  last two observations (p_prev NULL: zero velocity, :201-205)
 *   staleness      [n_q] or NULL (= 0)
 *   cur_pos        [n_q][P][2] or NULL: the t = 0 prepend of integrated_simulator.py:503-513 (skipped,
 *                  last step duplicated, when the first predicted step already equals it for every pedestrian)
 *   obs_float32    != 0: treat the observations as the float32 tensors the simulator's observer produces
 *                  (observer.py:131-132): positions rounded to float32, velocity a float32 quotient
 *   out            [n_q][P][T_out][2], T_out = n_steps + (cur_pos != NULL) */
int fot_predict_cv_device(int device, void* stream, int n_q, int P, const double* p_curr, const double* p_prev,
                          const double* staleness, double sgan_dt, const double* time_target, int n_steps,
                          const double* cur_pos, int obs_float32, double* out);

/* Replaces TrajectoryPredictor.process_prediction (:233-313) for S samples per query.
 *   pred   [n_q][S][pred_len][P][2]  raw predictor output (pred_len <= 64)
 *   anchor [n_q][P][2] or NULL       last observed positions (:277-279)
 *   out    [n_q][S][P][n_steps][2] */
int fot_process_prediction_device(int device, void* stream, int n_q, int S, int P, int pred_len, const double* pred,
                                  const double* anchor, const double* staleness, double sgan_dt,
                                  const double* time_target, int n_steps, double* out);

/* Replaces the closest-to-mean selection of TrajectoryPredictor.predict_single_best (:346-351).
 *   samples [n_q][S][P][T][2];  dist_scratch [n_q][S];  best_idx [n_q] */
int fot_select_best_sample_device(int device, void* stream, int n_q, int S, int P, int T, const double* samples,
                                  double* dist_scratch, int32_t* best_idx);

/* The t = 0 prepend of IntegratedSimulator._update_prediction (integrated_simulator.py:503-525).
 *   in   [n_q][S][P][T][2];  pick [n_q] or NULL (one sample per query: the representative sample)
 *   out  [n_q][pick ? 1 : S][P][T + 1][2]
 *   conditional != 0: the single-sample rule (:506-513); 0: the distribution rule (:517-525). */
int fot_prepend_current_device(int device, void* stream, int n_q, int S, int P, int T, const double* in,
                               const int32_t* pick, const double* cur_pos, int conditional, double* out);

/* ---- next row (SURVEY.md section 8f, rank 2): the state machine's inputs on the device -------------
 * Replaces compute_safety_metrics_static (src/core/data_structures.py:301-388) for n_q queries.
 *   ego      [n_q][5]      x, y, yaw, v, a
 *   ped_pos  [n_q][P][2], ped_vel [n_q][P][2];  n_peds [n_q] or NULL (= P for every query)
 *   combined_radius        ego_radius + ped_radius, or footprint.radius + ped_radius (:331-335)
 *   offsets  [n_circ]      HOST pointer, EgoFootprint.offsets (n_circ = 0: the centre circle)
 *   out      [n_q][5]      min_distance, collision (0 / 1), ttc, clearance, clearance_ahead (+inf = none) */
int fot_safety_metrics_device(int device, void* stream, int n_q, int P, const double* ego, const double* ped_pos,
                              const double* ped_vel, const int32_t* n_peds, double combined_radius,
                              const double* offsets, int n_circ, double* out);

/* ---- ego state -> Frenet: the nearest-point search on the device (DESIGN.md section 4e) -------------------------
 * best_s of find_nearest_point_on_path for n points (coordinate_converter.py:202-283) on the handle's path.
 * x, y, prev_s (NaN = no cache) [n], s_out [n], status [n]: DEVICE pointers; status 0 = s_out is the reference's
 * value, 1 = the caller must recompute that point on the host.  Asynchronous on `stream`, the stream on which the
 * inputs are written (NULL: the handle's stream, ordered after the work queued so far on the legacy default stream,
 * and synchronised).  prev_s is only read: the caller updates its caches. */
int fot_nearest_s_device(fot_handle_t* h, void* stream, int n, const double* x, const double* y,
                         const double* prev_s, double* s_out, int32_t* status);

#ifdef __cplusplus
}
#endif
#endif /* FOT_H_ */
