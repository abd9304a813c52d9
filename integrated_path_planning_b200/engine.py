"""Host side of the sweep: planner-constant tables, the fot handle, one launch per batch.

Everything numeric that the reference computes once per planner or once per call OUTSIDE the
candidate loops is built here with the reference's own NumPy expressions, so the kernel starts
from bit-identical grids, time tables and thresholds:
  horizon grid      frenet_planner.py:397-398      lateral grid   :419-420
  speed grid        :410-413                       brake ladder   :473-485
  TimeCache inverses :599-616 (numpy.linalg.inv)   collision radii :1172-1175
The candidate sweep itself runs only on the GPU (csrc/fot_kernels.cuh) through the C ABI.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import functools
import itertools
from dataclasses import dataclass
from typing import Any, Optional

import numpy as np

from . import _lib
from .spline import spline_tables
from .types import SERIES

BRAKE_T_MIN = 0.5
BRAKE_T_STEP = 0.5


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data


def horizon_grid(min_t, max_t, dt) -> np.ndarray:
    n_ti = int((max_t - min_t) / dt + 1e-9)
    return np.asarray(min_t + np.arange(n_ti + 1) * dt, dtype=np.float64)


def lateral_grid(d_road_w, max_road_width) -> np.ndarray:
    n_side = int(max_road_width / d_road_w + 1e-9)
    return np.asarray(np.arange(-n_side, n_side + 1) * d_road_w, dtype=np.float64)


def speed_grid(target_speed, d_t_s) -> np.ndarray:
    """One query's terminal-speed grid (frenet_planner.py:410-413)."""
    n_down = int(target_speed / d_t_s + 1e-9)
    if n_down < 0:
        raise ValueError("target_speed too negative for the speed grid")
    tv = target_speed - np.arange(n_down + 1) * d_t_s
    if tv[-1] > 1e-9:
        tv = np.append(tv, 0.0)
    return np.asarray(tv, dtype=np.float64)


def speed_grid_batch(target_speed: np.ndarray, d_t_s: float):
    """Vectorised speed_grid: returns (v_grid [n_q, n_v_max], n_v [n_q]); same elementwise
    arithmetic as the scalar version."""
    target = np.asarray(target_speed, dtype=np.float64).reshape(-1)
    if target.size > 1 and target.min() == target.max():
        # one target speed for the whole batch (the usual case): one row, repeated -- same arithmetic per element
        grid, n_v = speed_grid_batch(target[:1], d_t_s)
        return np.repeat(grid, target.size, axis=0), np.repeat(n_v, target.size)
    n_down = np.trunc(target / d_t_s + 1e-9).astype(np.int64)
    if np.any(n_down < 0):
        raise ValueError("target_speed too negative for the speed grid")
    width = int(n_down.max()) + 2
    k = np.arange(width)
    grid = target[:, None] - k[None, :] * d_t_s
    last = grid[np.arange(target.size), n_down]
    extra = last > 1e-9
    n_v = (n_down + 1 + extra).astype(np.int32)
    cols = np.arange(width)[None, :]
    grid = np.where(cols <= n_down[:, None], grid, 0.0)
    n_v_max = int(n_v.max())
    return np.ascontiguousarray(grid[:, :n_v_max]), n_v


def time_table(T, dt):
    """n_steps and the two inverse boundary matrices of one horizon (frenet_planner.py:593-616)."""
    n_steps = int(round(T / dt))
    ts = float(T)
    quartic = np.array([[3.0 * ts ** 2, 4.0 * ts ** 3],
                        [6.0 * ts, 12.0 * ts ** 2]])
    quintic = np.array([[ts ** 3, ts ** 4, ts ** 5],
                        [3.0 * ts ** 2, 4.0 * ts ** 3, 5.0 * ts ** 4],
                        [6.0 * ts, 12.0 * ts ** 2, 20.0 * ts ** 3]])
    return n_steps, np.linalg.inv(quartic), np.linalg.inv(quintic)


def winner_fields(n_t: int):
    """The winner block of fot_result_t as (name, torch dtype, per-query shape) with n_t samples per winner series, in
    the order of `WinnerBlock`'s sections: that order is the byte layout the gathers of the sharded sweep move."""
    import torch
    return (("best_idx", torch.int32, ()), ("winner_len", torch.int32, ()), ("stats", torch.int32, (_lib.FOT_N_STATS,)),
            ("best_cost", torch.float64, ()), ("winner", torch.float64, (_lib.FOT_N_SERIES, int(n_t))))


@dataclass
class QueryArrays:
    """A batch's inputs as fot_batch_t reads them (`query_arrays` builds and checks them)."""
    frenet: np.ndarray            # [n_q, 6]
    target: np.ndarray            # [n_q]
    limits: np.ndarray            # [n_q, 4]
    stop: np.ndarray              # [n_q], NaN = none
    v_grid: np.ndarray            # [n_q, n_v_max]
    n_v: np.ndarray               # [n_q] int32
    static: Optional[np.ndarray]  # [M, 2] shared or [n_q, M, 2] per query; None when empty
    static_per_query: bool
    dyn: Any                      # [n_q, S, P, T, 2] float64, a NumPy array or a CUDA torch tensor; None for FOT_DYN_NONE
    dyn_mode: int
    route: Optional[np.ndarray] = None   # [n_q] int32 route of every query (`route_array`); None: every query on route 0


def route_array(route, n_q: int, n_routes: int) -> Optional[np.ndarray]:
    """The per-query route ids of a batch as a contiguous int32 [n_q] array, from None (every query on route 0: returns
    None), one integer for every query, or [n_q] integers.  Raises ValueError on a non-integer value, a wrong shape or an
    id outside [0, n_routes): checked on the host, before anything reaches the device."""
    if route is None:
        return None
    a = np.asarray(route)
    if a.dtype == np.bool_ or not np.issubdtype(a.dtype, np.integer):
        raise ValueError(f"route must be integers, got {a.dtype}")
    if a.ndim == 0:
        a = np.full(n_q, a)
    elif a.shape != (n_q,):
        raise ValueError(f"route must be a scalar or [n_q={n_q}], got {list(a.shape)}")
    if a.size and (a.min() < 0 or a.max() >= n_routes):
        raise ValueError(f"route ids must be in [0, {n_routes}), got {int(a.min())}..{int(a.max())}")
    return np.ascontiguousarray(a, dtype=np.int32)


@functools.lru_cache(maxsize=8)
def _uniform_speed_grid(target_speed: float, n_q: int, d_t_s: float):
    return speed_grid_batch(np.full(n_q, target_speed), d_t_s)


def query_arrays(frenet, target_speed, limits, stop_dist, static, dyn, dyn_mode, d_t_s) -> QueryArrays:
    """A batch's inputs as QueryArrays, from target_speed and stop_dist (None: no stop distance) as scalars or [n_q],
    limits [4] or [n_q,4], and dyn as a NumPy array (converted) or a torch tensor.  Raises ValueError on a static or
    dyn of any other shape than QueryArrays lists: the C side reads them at the offsets those shapes give."""
    frenet = np.ascontiguousarray(frenet, dtype=np.float64).reshape(-1, 6)
    n_q = frenet.shape[0]
    full = lambda a, shape: np.array(np.broadcast_to(np.asarray(a, dtype=np.float64), shape), order="C")
    target = full(target_speed, (n_q,))
    if np.ndim(target_speed) == 0:      # one target speed for the whole batch (the usual case): an earlier call's grid
        v_grid, n_v = _uniform_speed_grid(float(target_speed), n_q, float(d_t_s))
    else:
        v_grid, n_v = speed_grid_batch(target, d_t_s)
    static = np.ascontiguousarray(static, dtype=np.float64) if static is not None and np.size(static) > 0 else None
    if static is not None and (static.ndim not in (2, 3) or static.shape[-1] != 2 or
                               (static.ndim == 3 and static.shape[0] != n_q)):
        raise ValueError(f"static obstacles must be [M, 2] or [n_q={n_q}, M, 2], got {list(static.shape)}")
    if dyn_mode == _lib.FOT_DYN_NONE:
        dyn = None
    else:
        if hasattr(dyn, "data_ptr"):                # a torch tensor stays where it is
            import torch
            dyn, f64 = dyn.contiguous(), torch.float64
        else:
            dyn, f64 = np.ascontiguousarray(dyn, dtype=np.float64), np.float64
        if dyn.ndim != 5 or dyn.shape[0] != n_q or dyn.shape[-1] != 2 or dyn.dtype != f64:
            raise ValueError(f"dyn must be float64 [n_q={n_q}, S, P, T, 2], got {dyn.dtype} {list(dyn.shape)}")
    return QueryArrays(frenet, target, full(limits, (n_q, 4)),
                       full(np.nan if stop_dist is None else stop_dist, (n_q,)), v_grid, n_v, static,
                       static is not None and static.ndim == 3, dyn, dyn_mode)


def fot_batch(q: QueryArrays, ptr) -> "_lib.FotBatch":
    """fot_batch_t over the arrays of q (host arrays or their device copies); ptr maps one to its address."""
    b = _lib.FotBatch()
    b.n_q, b.n_v_max = len(q.frenet), q.v_grid.shape[1]
    b.frenet, b.target_speed, b.limits, b.stop_dist = ptr(q.frenet), ptr(q.target), ptr(q.limits), ptr(q.stop)
    b.v_grid, b.n_v = ptr(q.v_grid), ptr(q.n_v)
    if q.static is not None:
        b.static_obs, b.n_static, b.static_per_query = ptr(q.static), q.static.shape[-2], int(q.static_per_query)
    if q.dyn is not None:
        b.dyn, b.dyn_mode = ptr(q.dyn), q.dyn_mode
        b.S, b.P, b.T_obs = q.dyn.shape[1], q.dyn.shape[2], q.dyn.shape[3]
    return b


# outputs of fot_assess_trajectories per (query, trajectory): (key, dtype name, trailing shape; "r" = n_r)
ASSESS_FIELDS = (("dyn_min", "float64", ()), ("dyn_at", "int32", (4,)), ("static_min", "float64", ()),
                 ("static_at", "int32", (3,)), ("dyn_hits", "int32", ("r",)), ("first_hit", "int32", ("r",)),
                 ("static_hit", "int32", ("r",)))


def assess_radii(r2) -> np.ndarray:
    """Threshold pairs (r2_dyn, r2_static) of fot_assess_trajectories as a contiguous float64 [n_r, 2] array, from one
    pair or [n_r, 2].  Raises ValueError on any other shape or n_r outside [1, FOT_MAX_RADII]."""
    a = np.ascontiguousarray(r2, dtype=np.float64)
    if a.ndim == 1:
        a = a.reshape(1, -1)
    if a.ndim != 2 or a.shape[1] != 2 or not 1 <= a.shape[0] <= _lib.FOT_MAX_RADII:
        raise ValueError(f"r2 must be one (r2_dyn, r2_static) pair or [n_r, 2] with n_r in [1, {_lib.FOT_MAX_RADII}], "
                         f"got {list(np.shape(r2))}")
    return a


def pack_paths(paths, n_t: Optional[int] = None):
    """A list of m FrenetPath-like objects (attributes named as types.SERIES) as the series block of one query:
    (series [m, 15, n_t] float64, NaN past each path's end; len [m] int32 = the samples of x).  n_t defaults to the
    longest path (at least 1).  Raises ValueError for m outside [1, FOT_MAX_ASSESSED] or a path longer than n_t or
    FOT_MAX_ASSESS_NT."""
    paths = list(paths)
    if not 1 <= len(paths) <= _lib.FOT_MAX_ASSESSED:
        raise ValueError(f"assess takes 1 to {_lib.FOT_MAX_ASSESSED} paths, got {len(paths)}")
    lens = np.array([len(getattr(p, "x")) for p in paths], dtype=np.int32)
    n_t = max(1, int(lens.max())) if n_t is None else int(n_t)
    if int(lens.max()) > n_t or n_t > _lib.FOT_MAX_ASSESS_NT:
        raise ValueError(f"paths of up to {_lib.FOT_MAX_ASSESS_NT} samples can be assessed, got {int(lens.max())}")
    series = np.full((len(paths), _lib.FOT_N_SERIES, n_t), np.nan)
    for j, p in enumerate(paths):
        for r, name in enumerate(SERIES):
            v = np.asarray(getattr(p, name, ()), dtype=np.float64).reshape(-1)[:lens[j]]
            series[j, r, :v.size] = v
    return series, lens


def fot_result(arrays, ptr, winner_samples: int = 0) -> "_lib.FotResult":
    """fot_result_t over the winner-block fields of arrays and, where not None, its cand_cat / cand_cost (addresses: ptr)."""
    r = _lib.FotResult()
    for name, _, _ in winner_fields(0):
        setattr(r, name, ptr(arrays[name]))
    if arrays.get("cand_cat") is not None:
        r.cand_cat, r.cand_stride = ptr(arrays["cand_cat"]), arrays["cand_cat"].shape[1]
    if arrays.get("cand_cost") is not None:
        r.cand_cost = ptr(arrays["cand_cost"])
    r.winner_samples = int(winner_samples)
    return r


@dataclass
class SweepResult:
    """Host copy of fot_result_t for n_q queries."""
    best_idx: np.ndarray      # [n_q] int32
    best_cost: np.ndarray     # [n_q]
    stats: np.ndarray         # [n_q, 8] int32, slot order _lib.STAT_KEYS
    winner_len: np.ndarray    # [n_q] int32
    winner: np.ndarray        # [n_q, 15, n_t_max]
    cand_cat: Optional[np.ndarray] = None    # [n_q, stride] uint8
    cand_cost: Optional[np.ndarray] = None   # [n_q, stride]
    n_cand: Optional[np.ndarray] = None      # [n_q] candidates generated per query
    kernel_ms: float = float("nan")
    # ranked alternatives (top_k > 0; include/fot.h fot_ranked_t): rank 0 is the winner, -1 / inf / 0 pad the ranks
    # past the last feasible candidate
    rank_idx: Optional[np.ndarray] = None     # [n_q, k] int32
    rank_cost: Optional[np.ndarray] = None    # [n_q, k]
    rank_len: Optional[np.ndarray] = None     # [n_q, k] int32, or None without series
    rank_series: Optional[np.ndarray] = None  # [n_q, k, 15, n_t_max], or None
    # winners under cost weightings (cost_weights; include/fot.h fot_weighted_t): -1 / inf / 0 where none is feasible
    w_idx: Optional[np.ndarray] = None        # [n_q, n_w] int32
    w_cost: Optional[np.ndarray] = None       # [n_q, n_w]
    w_len: Optional[np.ndarray] = None        # [n_q, n_w] int32, or None without series
    w_series: Optional[np.ndarray] = None     # [n_q, n_w, 15, n_t_max], or None
    cost_terms: Optional[np.ndarray] = None   # [n_q, stride, 5] (Jp, Jd, Js, Jv, Jt), NaN past the candidates
    # trajectory assessment (assess=True; include/fot.h fot_assessed_t): {name: array} for the names of ASSESS_FIELDS,
    # [n_q, m], [n_q, m, 4], [n_q, m, 3] or [n_q, m, n_r]; column 0 the winner, or with ranked series column j rank j.
    # A plain attribute, not a field: None unless the batch was assessed.
    assessed = None
    # candidate assessment (assess_candidates=True; include/fot.h fot_assess_candidates): the same names plus "keep",
    # [n_q, stride, ...], column i candidate i in generation order, blank past the query's candidates.  A plain
    # attribute: None unless the batch asked for it.
    cand_assessed = None

    def series(self, q: int = 0):
        """The 15 winner sequences of query q truncated to their kept length, or None."""
        if self.best_idx[q] < 0:
            return None
        n = min(int(self.winner_len[q]), self.winner.shape[2])      # winner_samples = k: the first k samples only
        return {name: self.winner[q, j, :n].copy() for j, name in enumerate(SERIES)}

    def alternatives(self, q: int = 0):
        """The ranked alternatives of query q, best first: a list of {"index", "cost", "series"}, where series holds
        the 15 sequences truncated to their kept length (None when the series were not requested)."""
        entries = (self._entry("rank", q, r) for r in range(self.rank_idx.shape[1]))
        return list(itertools.takewhile(lambda e: e is not None, entries))

    def under_weights(self, q: int = 0):
        """The winner of query q under each weighting, in weighting order: {"index", "cost", "series"} (series: the 15
        sequences truncated to their kept length, or None when they were not requested), or None where no candidate
        is feasible under that weighting."""
        return [self._entry("w", q, w) for w in range(self.w_idx.shape[1])]

    def assessment(self, q: int = 0):
        """The assessment of query q (a batch run with assess=True): {name: array} for the names of ASSESS_FIELDS, each
        with a leading dimension of one column per assessed trajectory -- column 0 the winner, or with ranked series
        column j rank j.  Blank columns (no winner, padded ranks) hold +inf, -1 and 0."""
        if self.assessed is None:
            raise ValueError("this result has no assessment: run the batch with assess=True")
        return {name: self.assessed[name][q].copy() for name, _, _ in ASSESS_FIELDS}

    def candidate_assessment(self, q: int = 0):
        """The assessment of every candidate of query q (a batch run with assess_candidates=True): {name: array} for
        the names of ASSESS_FIELDS and "keep" (samples assessed), one row per candidate in generation order, trimmed to
        the query's n_cand candidates; with "cand_cat" and "cand_cost" too when the candidate table was requested.
        Rows with keep 0 (emptied candidates, failed conversions) hold +inf, -1 and 0."""
        if self.cand_assessed is None:
            raise ValueError("this result has no candidate assessment: run the batch with assess_candidates=True")
        n = int(self.n_cand[q]) if self.n_cand is not None else self.cand_assessed["keep"].shape[1]
        out = {name: self.cand_assessed[name][q, :n].copy() for name in (*(f[0] for f in ASSESS_FIELDS), "keep")}
        for name in ("cand_cat", "cand_cost"):
            if getattr(self, name) is not None:
                out[name] = getattr(self, name)[q, :n].copy()
        return out

    def _entry(self, block: str, q: int, j: int):
        """Entry j of query q of the ranked ("rank") or weighted ("w") outputs, or None where its index is -1."""
        i = int(getattr(self, block + "_idx")[q, j])
        if i < 0:
            return None
        series, lens = getattr(self, block + "_series"), getattr(self, block + "_len")
        if series is not None:
            n = int(lens[q, j])
            series = {name: series[q, j, s, :n].copy() for s, name in enumerate(SERIES)}
        return {"index": i, "cost": np.float64(getattr(self, block + "_cost")[q, j]), "series": series}

    def blank(self, rows) -> None:
        """Queries `rows` (indices or a mask) as plan() returning None leaves them: index -1, cost inf, stats and kept
        lengths 0 in the winner, ranked and weighted outputs, cost terms NaN, assessments and candidate assessments
        blank (+inf, -1, 0, keep 0); the series and candidate table stay."""
        for name, value in (("best_idx", -1), ("best_cost", np.inf), ("stats", 0), ("winner_len", 0), ("rank_idx", -1),
                            ("rank_cost", np.inf), ("rank_len", 0), ("w_idx", -1), ("w_cost", np.inf), ("w_len", 0),
                            ("cost_terms", np.nan)):
            a = getattr(self, name)
            if a is not None:
                a[rows] = value
        for name, value in (("dyn_min", np.inf), ("dyn_at", -1), ("static_min", np.inf), ("static_at", -1),
                            ("dyn_hits", 0), ("first_hit", -1), ("static_hit", 0), ("keep", 0)):
            if self.assessed is not None and name in self.assessed:
                self.assessed[name][rows] = value
            if self.cand_assessed is not None:
                self.cand_assessed[name][rows] = value


class SweepEngine:
    """Owns one fot handle (one device).  Built from the planner's constructor knobs."""

    def __init__(self, reference_path, *, max_speed, dt, d_road_w, max_road_width, robot_radius,
                 obstacle_radius, min_t, max_t, k_j, k_t, k_d, k_s_dot, k_lat, k_lon,
                 chance_epsilon=0.0, collision_margin_inflation=1.0, footprint=None, device=0):
        self.lib = _lib.load()
        self.device = int(device)
        self.dt = dt
        sp = spline_tables(reference_path)

        T = horizon_grid(min_t, max_t, dt)
        tabs = [time_table(t, dt) for t in T]
        d_grid = lateral_grid(d_road_w, max_road_width)
        if T.size == 0 or d_grid.size == 0:
            raise ValueError("empty horizon or lateral grid")
        n_total = int(round(max_t / dt)) + 1
        Tb_all = np.arange(BRAKE_T_MIN, min_t - 1e-9, BRAKE_T_STEP)
        btabs = [(tb, *time_table(tb, dt)) for tb in Tb_all]
        btabs = [b for b in btabs if n_total - (b[1] + 1) >= 0]      # :483-485 n_pad < 0 -> skipped

        if footprint is None:
            ego_radius = robot_radius
            offsets = np.zeros(0)
        else:
            ego_radius = footprint.radius
            offsets = np.asarray(footprint.offsets, dtype=np.float64).reshape(-1)
            if offsets.size > _lib.FOT_MAX_CIRCLES or offsets.size == 0:
                raise ValueError(f"footprint with {offsets.size} circles unsupported (1..{_lib.FOT_MAX_CIRCLES})")
        inflated_radius = max(ego_radius + obstacle_radius, 1e-6)
        dyn_radius = inflated_radius * collision_margin_inflation
        sq_rubicon = inflated_radius ** 2
        sq_rubicon_dyn = dyn_radius ** 2
        self.collide_r2, self.collide_r2_single, self.chance_epsilon = sq_rubicon, sq_rubicon_dyn, float(chance_epsilon)

        cfg = _lib.FotConfig()
        cfg.dt, cfg.max_speed, cfg.max_road_width = dt, max_speed, max_road_width
        cfg.k_j, cfg.k_t, cfg.k_d, cfg.k_s_dot, cfg.k_lat, cfg.k_lon = k_j, k_t, k_d, k_s_dot, k_lat, k_lon
        cfg.collide_r2, cfg.collide_r2_single, cfg.chance_epsilon = sq_rubicon, sq_rubicon_dyn, chance_epsilon
        for i, o in enumerate(offsets):
            cfg.circle_offsets[i] = float(o)
        cfg.n_circles = int(offsets.size)
        cfg.n_T, cfg.n_d, cfg.n_B, cfg.n_total, cfg.nx = len(T), len(d_grid), len(btabs), n_total, len(sp["knots"])

        f64 = lambda seq, shape: np.ascontiguousarray(np.array(seq, dtype=np.float64).reshape(shape))
        i32 = lambda seq: np.ascontiguousarray(np.array(seq, dtype=np.int32).reshape(-1))
        self._keep = {                                     # keep host arrays alive during create
            "T": f64(T, (-1,)), "n_steps": i32([t[0] for t in tabs]),
            "inv4": f64([t[1] for t in tabs], (-1,)), "inv5": f64([t[2] for t in tabs], (-1,)),
            "Tb": f64([b[0] for b in btabs], (-1,)), "n_steps_b": i32([b[1] for b in btabs]),
            "inv4b": f64([b[2] for b in btabs], (-1,)), "inv5b": f64([b[3] for b in btabs], (-1,)),
            "d_grid": f64(d_grid, (-1,)), **sp,
        }
        tb = _lib.FotTables()
        for name, _ in _lib.FotTables._fields_:
            arr = self._keep[name]
            ctype = _lib.c_int32_p if arr.dtype == np.int32 else _lib.c_double_p
            setattr(tb, name, arr.ctypes.data_as(ctype) if arr.size else None)
        self.n_T, self.n_d, self.n_B = cfg.n_T, cfg.n_d, cfg.n_B
        self.n_circles = int(cfg.n_circles)
        self.T, self.d_grid, self.Tb = self._keep["T"], self._keep["d_grid"], self._keep["Tb"]
        self.n_steps, self.n_steps_b, self.n_total = self._keep["n_steps"], self._keep["n_steps_b"], n_total
        self._pinned = {}
        self._near_bufs = None                             # nearest_s: pinned / device staging, grown on demand
        self._near_stream = None                           # nearest_s: its stream
        self._h = C.c_void_p()
        _lib.check(self.lib.fot_create(C.byref(cfg), C.byref(tb), self.device, C.byref(self._h)), "fot_create")
        self.n_t_max = self.lib.fot_n_t_max(self._h)

    def add_route(self, path) -> int:
        """Registers one more reference path (a CubicSpline2D or the reference's spline object) on the device: its id
        (1, 2, ...) is what the route arrays of the batch calls name.  Route 0 is the path of the constructor."""
        sp = spline_tables(path)
        self._keep.setdefault("routes", []).append(sp)      # host tables stay alive with the engine
        r = _lib.FotRoute(nx=len(sp["knots"]))
        for name, _ in _lib.FotRoute._fields_[1:]:
            setattr(r, name, sp[name].ctypes.data_as(_lib.c_double_p))
        rid = C.c_int32()
        _lib.check(self.lib.fot_add_route(self._h, C.byref(r), C.byref(rid)), "fot_add_route")
        return int(rid.value)

    @contextlib.contextmanager
    def routes_bound(self, route_ptr: Optional[int]):
        """The calls inside the block plan query q on the route in route_ptr[q] (a device int32 array; fot_set_routes);
        the binding is cleared on leaving, so none outlives the block.  None: no binding."""
        if route_ptr is None:
            yield
            return
        _lib.check(self.lib.fot_set_routes(self._h, C.c_void_p(route_ptr)), "fot_set_routes")
        try:
            yield
        finally:
            self.lib.fot_set_routes(self._h, None)

    def close(self):
        if getattr(self, "_h", None):
            self.lib.fot_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---------------------------------------------------------------------------------
    def candidate_counts(self, frenet: np.ndarray, n_v: np.ndarray) -> np.ndarray:
        has_brake = (frenet[:, 1] > 0.1) & (self.n_B > 0)
        return (self.n_T * n_v.astype(np.int64) * self.n_d + has_brake * self.n_B).astype(np.int64)

    def points_per_query(self, frenet: np.ndarray, n_v: np.ndarray) -> np.ndarray:
        """Un-truncated trajectory samples per query (the E of SURVEY.md section 8d divides by this)."""
        per_T = (self.n_steps.astype(np.int64) + 1).sum()
        has_brake = (frenet[:, 1] > 0.1) & (self.n_B > 0)
        return per_T * n_v.astype(np.int64) * self.n_d + has_brake * self.n_B * self.n_total

    def run_host(self, q: QueryArrays, want_candidates=False, winner_samples: int = 0) -> SweepResult:
        """One fot_plan_batch_host call on the host arrays of q.  winner_samples = k > 0: only the first k samples
        of each winner series come back (`winner` is [n_q,15,k]); `fetch_winners` reads full series of the last
        call from the device."""
        k_head = min(int(winner_samples), self.n_t_max) if winner_samples and winner_samples > 0 else 0
        res = self._result_buffers(len(q.frenet), want_candidates, q.v_grid.shape[1], k_head)
        b, r = fot_batch(q, _ptr), fot_result(vars(res), _ptr, k_head)
        route_d = self._device_route(q.route)                # the route array is device memory for this call too
        with self.routes_bound(None if route_d is None else route_d.data_ptr()):
            _lib.check(self.lib.fot_plan_batch_host(self._h, C.byref(b), C.byref(r)), "fot_plan_batch_host")
        return self.finish_result(res, q.frenet, q.n_v)

    def _device_route(self, route: Optional[np.ndarray]):
        """A route array (`route_array`) as an int32 tensor on this engine's device, or None."""
        if route is None:
            return None
        import torch
        return torch.from_numpy(np.ascontiguousarray(route, dtype=np.int32)).to(torch.device("cuda", self.device))

    def finish_result(self, res: SweepResult, frenet: np.ndarray, n_v: np.ndarray) -> SweepResult:
        """res with the candidates generated per query and the device time of the last launch filled in."""
        res.n_cand = self.candidate_counts(frenet, n_v)
        res.kernel_ms = self.last_kernel_ms()
        return res

    def fetch_winners(self, q0: int, n: int) -> np.ndarray:
        """Full winner series [n,15,n_t_max] of queries q0..q0+n-1 of the last run_host call (fot_fetch_winners)."""
        out = np.empty((n, _lib.FOT_N_SERIES, self.n_t_max), dtype=np.float64)
        _lib.check(self.lib.fot_fetch_winners(self._h, int(q0), int(n), _ptr(out)), "fot_fetch_winners")
        return out

    def reload_options(self) -> None:
        """Re-read the FOT_* tuning environment for this handle (tests / tuning; the planning calls never read it)."""
        _lib.check(self.lib.fot_reload_options(self._h), "fot_reload_options")

    def _result_buffers(self, n_q: int, want_candidates: bool, n_v_max: int, k_head: int = 0) -> SweepResult:
        """Result arrays in pinned host memory (torch is only the allocator), cached per batch size so
        the device->host copies are true async DMAs.  The arrays of a returned SweepResult stay valid
        until the next call on this engine with the same batch size."""
        import torch
        stride = self.lib.fot_candidate_count(self._h, n_v_max, 1) if want_candidates else 0
        key = (n_q, stride, k_head)
        cached = self._pinned.get(key)
        if cached is None:
            pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True).numpy()
            cached = {name: pin((n_q, *shape), dt) for name, dt, shape in winner_fields(k_head or self.n_t_max)}
            if want_candidates:
                cached["cand_cat"] = pin((n_q, stride), torch.uint8)
                cached["cand_cost"] = pin((n_q, stride), torch.float64)
            if len(self._pinned) > 8:
                self._pinned.clear()
            self._pinned[key] = cached
        return SweepResult(**cached)

    def run_device(self, batch: "_lib.FotBatch", result: "_lib.FotResult", stream=None) -> None:
        """fot_plan_batch_device with caller-owned device pointers (torch tensors as buffers)."""
        _lib.check(self.lib.fot_plan_batch_device(self._h, C.byref(batch), C.byref(result),
                                                  C.c_void_p(stream) if stream else None),
                   "fot_plan_batch_device")

    def rank_device(self, batch: "_lib.FotBatch", cand_cat: int, cand_cost: int, cand_stride: int,
                    ranked: "_lib.FotRanked", stream=None) -> None:
        """fot_rank_candidates on the per-candidate table of a fot_plan_batch_device launch of `batch` (device
        pointers), stream-ordered behind it."""
        _lib.check(self.lib.fot_rank_candidates(self._h, C.byref(batch), C.c_void_p(cand_cat), C.c_void_p(cand_cost),
                                                int(cand_stride), C.byref(ranked), C.c_void_p(stream) if stream else None),
                   "fot_rank_candidates")

    def select_weighted_device(self, batch: "_lib.FotBatch", cand_cat: int, cand_stride: int,
                               weighted: "_lib.FotWeighted", stream=None) -> None:
        """fot_select_weighted on the per-candidate table of a fot_plan_batch_device launch of `batch` (device
        pointers), stream-ordered behind it."""
        _lib.check(self.lib.fot_select_weighted(self._h, C.byref(batch), C.c_void_p(cand_cat), int(cand_stride),
                                                C.byref(weighted), C.c_void_p(stream) if stream else None),
                   "fot_select_weighted")

    def cost_terms_device(self, batch: "_lib.FotBatch", cand_stride: int, terms: int, stream=None) -> None:
        """fot_cost_terms: (Jp, Jd, Js, Jv, Jt) of every candidate of `batch` into terms [n_q, cand_stride, 5]."""
        _lib.check(self.lib.fot_cost_terms(self._h, C.byref(batch), int(cand_stride), C.c_void_p(terms),
                                           C.c_void_p(stream) if stream else None), "fot_cost_terms")

    def own_radii(self, dyn_mode: int) -> np.ndarray:
        """This handle's own threshold pair [1, 2] for a field of dyn_mode: (collide_r2_single, collide_r2) for a single
        sample, (collide_r2, collide_r2) otherwise -- under it fot_assess_trajectories reproduces the collision verdict."""
        r2d = self.collide_r2_single if dyn_mode == _lib.FOT_DYN_SINGLE else self.collide_r2
        return np.array([[r2d, self.collide_r2]], dtype=np.float64)

    def assess_device(self, obstacles: "_lib.FotBatch", assessed: "_lib.FotAssessed", stream=None) -> None:
        """fot_assess_trajectories: the trajectories of `assessed` against the field of `obstacles` (device pointers),
        stream-ordered behind the launch that wrote their series."""
        _lib.check(self.lib.fot_assess_trajectories(self._h, C.byref(obstacles), C.byref(assessed),
                                                    C.c_void_p(stream) if stream else None), "fot_assess_trajectories")

    def assess_candidates_device(self, queries: "_lib.FotBatch", field: "_lib.FotBatch", cand_stride: int,
                                 assessed: "_lib.FotAssessed", keep: Optional[int] = None, stream=None) -> None:
        """fot_assess_candidates: every generated candidate of `queries` (device pointers) regenerated on the device and
        assessed against the field of `field` into the [n_q, cand_stride, ...] outputs of `assessed` (series and len
        null) and keep [n_q, cand_stride] (or None).  Needs no sweep."""
        _lib.check(self.lib.fot_assess_candidates(self._h, C.byref(queries), C.byref(field), int(cand_stride),
                                                  C.byref(assessed), C.c_void_p(keep) if keep else None,
                                                  C.c_void_p(stream) if stream else None), "fot_assess_candidates")

    def nearest_s(self, x, y, prev_s, route=None):
        """fot_nearest_s_device for m points on this engine's path (route: [m] route ids, point k on route[k]): returns
        (s [m], status [m] int32), status 0 where s is the reference's best_s, 1 where the host has to recompute it.
        One upload of x | y | prev_s, one download of s | status, one synchronise; prev_s (NaN = no cache) is not
        modified."""
        import torch
        m = len(x)
        if m == 0:
            return np.zeros(0), np.zeros(0, dtype=np.int32)
        bufs = self._near_bufs
        if bufs is None or bufs[0].numel() < 3 * m:
            cap = max(3 * m, 3 * 256)
            dev = torch.device("cuda", self.device)
            bufs = self._near_bufs = (torch.empty(cap, dtype=torch.float64, pin_memory=True),
                                      torch.empty(cap, dtype=torch.float64, device=dev),
                                      torch.empty(12 * (cap // 3), dtype=torch.uint8, pin_memory=True),
                                      torch.empty(12 * (cap // 3), dtype=torch.uint8, device=dev))
        h_in, d_in, h_out, d_out = bufs
        a = h_in.numpy()
        a[:m], a[m:2 * m], a[2 * m:3 * m] = x, y, prev_s
        # upload, kernel and download on one stream of this engine's own: the kernel is ordered after the upload
        # whatever stream the caller has made current (torch's default stream would reach the C call as NULL)
        if self._near_stream is None:
            self._near_stream = torch.cuda.Stream(self.device)
        stream = self._near_stream
        with torch.cuda.stream(stream):
            d_in[:3 * m].copy_(h_in[:3 * m], non_blocking=True)
            route_d = None if route is None else \
                torch.from_numpy(np.ascontiguousarray(route, dtype=np.int32)).to(d_in.device, non_blocking=False)
            p_in, p_out = d_in.data_ptr(), d_out.data_ptr()
            with self.routes_bound(None if route_d is None else route_d.data_ptr()):
                _lib.check(self.lib.fot_nearest_s_device(self._h, C.c_void_p(stream.cuda_stream), m, C.c_void_p(p_in),
                                                         C.c_void_p(p_in + 8 * m), C.c_void_p(p_in + 16 * m),
                                                         C.c_void_p(p_out), C.c_void_p(p_out + 8 * m)),
                           "fot_nearest_s_device")
            h_out[:12 * m].copy_(d_out[:12 * m], non_blocking=True)
        stream.synchronize()
        raw = h_out.numpy()
        return raw[:8 * m].view(np.float64).copy(), raw[8 * m:12 * m].view(np.int32).copy()

    def launch_stage_ms(self, back: int = 0):
        """(prepass, sweep, winner) device ms of the `back`-th most recent launch."""
        ms = (C.c_float * 3)()
        _lib.check(self.lib.fot_launch_stage_ms(self._h, int(back), C.byref(ms)), "fot_launch_stage_ms")
        return tuple(float(v) for v in ms)

    def last_kernel_ms(self) -> float:
        return float(self.lib.fot_last_kernel_ms(self._h))
