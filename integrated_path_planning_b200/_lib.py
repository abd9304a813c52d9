"""ctypes binding of the C ABI in include/fot.h (libfot.so, built in-tree by build.py).

Loading fails loudly: there is no CPU fallback and no JIT -- `build.py` (or
`__graft_entry__.build()`) must have produced `libfot.so` next to this file.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libfot.so")

FOT_ABI_VERSION = 8
FOT_ABI_MINOR = 1
FOT_MAX_CIRCLES = 8
FOT_MAX_RANKED = 32
FOT_MAX_WEIGHT_SETS = 256
FOT_MAX_ASSESSED = 256
FOT_MAX_RADII = 16
FOT_MAX_ASSESS_NT = 320
FOT_N_STATS = 8
FOT_N_SERIES = 15
FOT_DYN_NONE, FOT_DYN_SINGLE, FOT_DYN_DISTRIBUTION = 0, 1, 2
CAT_OK, CAT_SPEED, CAT_ACCEL, CAT_CURV, CAT_LAT, CAT_ROAD, CAT_COLL, CAT_STOP, CAT_DROP = range(9)
# last_check_stats keys in the slot order of fot_result_t.stats (frenet_planner.py:910-918, :324)
STAT_KEYS = ("ok", "max_speed_error", "max_accel_error", "max_curvature_error", "max_lat_accel_error",
             "road_bound_error", "collision_error", "stop_distance_error")
# the six cost weights in the order of fot_weighted_t.weights (frenet_planner.py:187-192)
COST_WEIGHT_KEYS = ("k_j", "k_t", "k_d", "k_s_dot", "k_lat", "k_lon")

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_uint8_p = C.POINTER(C.c_uint8)


class FotConfig(C.Structure):
    _fields_ = [
        ("dt", C.c_double), ("max_speed", C.c_double), ("max_road_width", C.c_double),
        ("k_j", C.c_double), ("k_t", C.c_double), ("k_d", C.c_double),
        ("k_s_dot", C.c_double), ("k_lat", C.c_double), ("k_lon", C.c_double),
        ("collide_r2", C.c_double), ("collide_r2_single", C.c_double), ("chance_epsilon", C.c_double),
        ("circle_offsets", C.c_double * FOT_MAX_CIRCLES),
        ("n_circles", C.c_int32), ("n_T", C.c_int32), ("n_d", C.c_int32), ("n_B", C.c_int32),
        ("n_total", C.c_int32), ("nx", C.c_int32),
    ]


class FotTables(C.Structure):
    _fields_ = [
        ("T", c_double_p), ("n_steps", c_int32_p), ("inv4", c_double_p), ("inv5", c_double_p),
        ("Tb", c_double_p), ("n_steps_b", c_int32_p), ("inv4b", c_double_p), ("inv5b", c_double_p),
        ("d_grid", c_double_p), ("knots", c_double_p),
        ("xa", c_double_p), ("xb", c_double_p), ("xc", c_double_p), ("xd", c_double_p),
        ("ya", c_double_p), ("yb", c_double_p), ("yc", c_double_p), ("yd", c_double_p),
    ]


class FotBatch(C.Structure):
    _fields_ = [
        ("n_q", C.c_int32), ("n_v_max", C.c_int32),
        ("frenet", C.c_void_p), ("target_speed", C.c_void_p), ("limits", C.c_void_p),
        ("stop_dist", C.c_void_p), ("v_grid", C.c_void_p), ("n_v", C.c_void_p),
        ("static_obs", C.c_void_p), ("n_static", C.c_int32), ("static_per_query", C.c_int32),
        ("dyn", C.c_void_p), ("S", C.c_int32), ("P", C.c_int32), ("T_obs", C.c_int32), ("dyn_mode", C.c_int32),
    ]


class FotResult(C.Structure):
    _fields_ = [
        ("best_idx", C.c_void_p), ("best_cost", C.c_void_p), ("stats", C.c_void_p),
        ("winner_len", C.c_void_p), ("winner", C.c_void_p),
        ("cand_cat", C.c_void_p), ("cand_cost", C.c_void_p),
        ("cand_stride", C.c_int32), ("winner_samples", C.c_int32),
    ]


class FotRanked(C.Structure):
    _fields_ = [
        ("k", C.c_int32), ("idx", C.c_void_p), ("cost", C.c_void_p), ("len", C.c_void_p), ("series", C.c_void_p),
    ]


class FotWeighted(C.Structure):
    _fields_ = [
        ("n_w", C.c_int32), ("per_query", C.c_int32), ("weights", C.c_void_p), ("idx", C.c_void_p),
        ("cost", C.c_void_p), ("len", C.c_void_p), ("series", C.c_void_p),
    ]


class FotAssessed(C.Structure):
    _fields_ = [
        ("m", C.c_int32), ("n_t", C.c_int32), ("n_r", C.c_int32),
        ("series", C.c_void_p), ("len", C.c_void_p), ("r2", C.c_void_p),
        ("dyn_min", C.c_void_p), ("dyn_at", C.c_void_p), ("static_min", C.c_void_p), ("static_at", C.c_void_p),
        ("dyn_hits", C.c_void_p), ("first_hit", C.c_void_p), ("static_hit", C.c_void_p),
    ]


class FotRoute(C.Structure):
    _fields_ = [
        ("nx", C.c_int32), ("knots", c_double_p),
        ("xa", c_double_p), ("xb", c_double_p), ("xc", c_double_p), ("xd", c_double_p),
        ("ya", c_double_p), ("yb", c_double_p), ("yc", c_double_p), ("yd", c_double_p),
    ]


# every symbol include/fot.h declares: (name, restype, argtypes)
SYMBOLS = (
    ("fot_abi_version", C.c_int, ()),
    ("fot_abi_minor", C.c_int, ()),
    ("fot_last_error", C.c_char_p, ()),
    ("fot_create", C.c_int, (C.POINTER(FotConfig), C.POINTER(FotTables), C.c_int, C.POINTER(C.c_void_p))),
    ("fot_destroy", C.c_int, (C.c_void_p,)),
    ("fot_n_t_max", C.c_int, (C.c_void_p,)),
    ("fot_candidate_count", C.c_int, (C.c_void_p, C.c_int, C.c_int)),
    ("fot_plan_batch_device", C.c_int, (C.c_void_p, C.POINTER(FotBatch), C.POINTER(FotResult), C.c_void_p)),
    ("fot_rank_candidates", C.c_int, (C.c_void_p, C.POINTER(FotBatch), C.c_void_p, C.c_void_p, C.c_int,
                                      C.POINTER(FotRanked), C.c_void_p)),
    ("fot_select_weighted", C.c_int, (C.c_void_p, C.POINTER(FotBatch), C.c_void_p, C.c_int, C.POINTER(FotWeighted),
                                      C.c_void_p)),
    ("fot_cost_terms", C.c_int, (C.c_void_p, C.POINTER(FotBatch), C.c_int, C.c_void_p, C.c_void_p)),
    ("fot_plan_batch_host", C.c_int, (C.c_void_p, C.POINTER(FotBatch), C.POINTER(FotResult))),
    ("fot_plan_batch_device_to_host", C.c_int, (C.c_void_p, C.POINTER(FotBatch), C.POINTER(FotResult), C.c_void_p)),
    ("fot_set_result_mirror", C.c_int, (C.c_void_p, C.POINTER(FotResult), C.c_void_p)),
    ("fot_peer_alloc", C.c_int, (C.c_int, C.c_size_t, C.POINTER(C.c_void_p), C.c_char_p)),
    ("fot_peer_open", C.c_int, (C.c_int, C.c_char_p, C.POINTER(C.c_void_p))),
    ("fot_peer_close", C.c_int, (C.c_void_p,)),
    ("fot_peer_free", C.c_int, (C.c_void_p,)),
    ("fot_peer_await", C.c_int, (C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_void_p)),
    ("fot_fetch_winners", C.c_int, (C.c_void_p, C.c_int, C.c_int, C.c_void_p)),
    ("fot_reload_options", C.c_int, (C.c_void_p,)),
    ("fot_last_kernel_ms", C.c_float, (C.c_void_p,)),
    ("fot_last_sweep_kind", C.c_int, (C.c_void_p,)),
    ("fot_last_pair_features", C.c_int, (C.c_void_p,)),
    ("fot_launch_stage_ms", C.c_int, (C.c_void_p, C.c_int, C.POINTER(C.c_float * 3))),
    ("fot_probe_fma_tflops", C.c_int, (C.c_int, C.c_int, c_double_p)),
    ("fot_predict_cv_device", C.c_int, (C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_double, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p)),
    ("fot_process_prediction_device", C.c_int, (C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_int, C.c_void_p)),
    ("fot_select_best_sample_device", C.c_int, (C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                C.c_void_p, C.c_void_p)),
    ("fot_prepend_current_device", C.c_int, (C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_int, C.c_void_p)),
    ("fot_safety_metrics_device", C.c_int, (C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_double, c_double_p, C.c_int, C.c_void_p)),
    ("fot_nearest_s_device", C.c_int, (C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p)),
    ("fot_add_route", C.c_int, (C.c_void_p, C.POINTER(FotRoute), C.POINTER(C.c_int32))),
    ("fot_set_routes", C.c_int, (C.c_void_p, C.c_void_p)),
    ("fot_assess_trajectories", C.c_int, (C.c_void_p, C.POINTER(FotBatch), C.POINTER(FotAssessed), C.c_void_p)),
    ("fot_assess_candidates", C.c_int, (C.c_void_p, C.POINTER(FotBatch), C.POINTER(FotBatch), C.c_int,
                                        C.POINTER(FotAssessed), C.c_void_p, C.c_void_p)),
)

_lib = None


class FotError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libfot.so and bind every exported symbol.  Raises FotError if the library has not
    been built -- the planner never falls back to a CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FotError(
            f"{LIB_PATH} is missing: build the CUDA library first "
            "(`python -m integrated_path_planning_b200.build` or `__graft_entry__.build()`); "
            "there is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, restype, argtypes in SYMBOLS:
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise FotError(f"libfot.so lacks {name} (built from older sources); rebuild") from None
        fn.restype = restype
        fn.argtypes = list(argtypes)
    if lib.fot_abi_version() != FOT_ABI_VERSION or lib.fot_abi_minor() != FOT_ABI_MINOR:
        raise FotError("libfot.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().fot_last_error()
        raise FotError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")
