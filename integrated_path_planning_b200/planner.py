"""Drop-in `FrenetPlanner`: the reference planner's Python API over the B200 sweep.

Same constructor, `plan()` signature, attributes and side effects as reference
`src/planning/frenet_planner.py:125-332` (see SURVEY.md section 8b), so it can be handed to the
reference's `IntegratedSimulator` in place of the NumPy planner
(`integrated_simulator.py:342-366, 576-584, 622-630, 800-802`).  What runs where:

  host (this file, O(1) per call)   ego -> Frenet state, constraint overrides, grids, FrenetPath
  GPU  (csrc/, via include/fot.h)   candidate generation, Frenet->global, validity chain,
                                    collision tests, cost, arg-min, winner regeneration

There is no CPU path for the sweep: without libfot.so or a CUDA device `plan()` raises.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import numpy as np

from . import _lib
from .engine import ASSESS_FIELDS, QueryArrays, SweepEngine, SweepResult, assess_radii, pack_paths, query_arrays
from .spline import spline_tables
from .frenet_host import CoordinateConverter, ego_to_frenet
from .types import FrenetPath, FrenetState, SERIES

# module defaults of the reference (frenet_planner.py:25-43, :91)
MAX_SPEED = 50.0 / 3.6
MAX_ACCEL = 2.0
MAX_CURVATURE = 1.0
MAX_ROAD_WIDTH = 7.0
D_ROAD_W = 0.5
DT = 0.2
MAX_T = 5.0
MIN_T = 4.0
TARGET_SPEED = 30.0 / 3.6
D_T_S = 5.0 / 3.6
N_S_SAMPLE = 1
K_J = 0.1
K_T = 0.1
K_D = 1.0
K_S_DOT = 1.0
K_LAT = 1.0
K_LON = 1.0
ROBOT_RADIUS = 2.0
MAX_LAT_ACCEL = 3.0

_REF_STAT_ORDER = ("max_speed_error", "max_accel_error", "max_curvature_error", "max_lat_accel_error",
                   "road_bound_error", "collision_error", "ok")


def _default_device() -> int:
    return int(os.environ.get("LOCAL_RANK", "0"))


def _frenet_path(series, cost) -> FrenetPath:
    """A FrenetPath from the 15 sequences of one candidate, as the reference returns it (frenet_planner.py:294)."""
    path = FrenetPath(cost=np.float64(cost))
    for name in SERIES[:9]:
        setattr(path, name, series[name])
    for name in SERIES[9:]:
        setattr(path, name, series[name].tolist())
    return path


def classify_dynamic(dynamic_obstacles, distribution):
    """Which dynamic-obstacle tensor the reference would use (frenet_planner.py:1043-1047,
    :1205-1208) -> (mode, array [1,S,P,T,2] or None)."""
    if distribution is not None and np.size(distribution) > 0:
        dist = np.asarray(distribution, dtype=np.float64)
        if dist.ndim == 4 and dist.shape[-1] == 2 and dist.shape[1] > 0 and dist.shape[2] > 0:
            return _lib.FOT_DYN_DISTRIBUTION, dist[None]
        return _lib.FOT_DYN_NONE, None       # every per-sample test returns False (:1205-1208)
    if dynamic_obstacles is not None and np.size(dynamic_obstacles) > 0:
        dyn = np.asarray(dynamic_obstacles, dtype=np.float64)
        if dyn.ndim == 3 and dyn.shape[-1] == 2:
            return _lib.FOT_DYN_SINGLE, dyn[None, None]
    return _lib.FOT_DYN_NONE, None


class FrenetPlanner:
    """Frenet optimal-trajectory planner (Werling et al. 2010) -- B200 candidate sweep."""

    SINGULARITY_EPS = 0.05
    EPS_S_DOT = 1e-3

    def __init__(self, reference_path, max_speed: float = MAX_SPEED, max_accel: float = MAX_ACCEL,
                 max_curvature: float = MAX_CURVATURE, dt: float = DT, d_road_w: float = D_ROAD_W,
                 max_road_width: float = MAX_ROAD_WIDTH, robot_radius: float = ROBOT_RADIUS,
                 obstacle_radius: float = 0.3, min_t: float = MIN_T, max_t: float = MAX_T,
                 d_t_s: float = D_T_S, n_s_sample: int = N_S_SAMPLE, **kwargs):
        self.csp = reference_path
        self.routes = [reference_path]           # route r of the batch calls (add_route); route 0 is this path
        self.max_speed = max_speed
        self.max_accel = max_accel
        self.max_curvature = max_curvature
        self.max_lat_accel = float(kwargs.get("max_lat_accel", MAX_LAT_ACCEL))
        self.dt = dt
        self.d_road_w = d_road_w
        self.max_road_width = max_road_width
        self.converter = CoordinateConverter(reference_path)
        self.robot_radius = robot_radius
        self.obstacle_radius = obstacle_radius
        self.min_t = min_t
        self.max_t = max_t
        self.d_t_s = d_t_s
        self.n_s_sample = n_s_sample            # accepted, unused (frenet_planner.py:401-403)
        self.k_j = kwargs.get("k_j", K_J)
        self.k_t = kwargs.get("k_t", K_T)
        self.k_d = kwargs.get("k_d", K_D)
        self.k_s_dot = kwargs.get("k_s_dot", K_S_DOT)
        self.k_lat = kwargs.get("k_lat", K_LAT)
        self.k_lon = kwargs.get("k_lon", K_LON)
        self.chance_epsilon = float(kwargs.get("chance_epsilon", 0.0))
        self.collision_margin_inflation = float(kwargs.get("collision_margin_inflation", 1.0))
        self.footprint = kwargs.get("footprint", None)
        self.device = int(kwargs.get("device", _default_device()))
        self._last_kappa = 0.0
        self.last_check_stats: Optional[Dict[str, int]] = None
        self.last_result: Optional[SweepResult] = None   # diagnostics: raw C-ABI output of the last call
        self._engine: Optional[SweepEngine] = None

    # -- engine ----------------------------------------------------------------------------
    @property
    def engine(self) -> SweepEngine:
        """The device handle, created on first use (so the host-side API can be exercised on a
        machine without a GPU; the sweep itself cannot)."""
        if self._engine is None:
            self._engine = SweepEngine(
                self.csp, max_speed=self.max_speed, dt=self.dt, d_road_w=self.d_road_w,
                max_road_width=self.max_road_width, robot_radius=self.robot_radius,
                obstacle_radius=self.obstacle_radius, min_t=self.min_t, max_t=self.max_t,
                k_j=self.k_j, k_t=self.k_t, k_d=self.k_d, k_s_dot=self.k_s_dot, k_lat=self.k_lat,
                k_lon=self.k_lon, chance_epsilon=self.chance_epsilon,
                collision_margin_inflation=self.collision_margin_inflation, footprint=self.footprint,
                device=self.device)
            for path in self.routes[1:]:
                self._engine.add_route(path)
        return self._engine

    def add_route(self, reference_path) -> int:
        """One more reference path (a CubicSpline2D or the reference's spline object) for the batch calls, which take a
        `route` per query; returns its id, the index into `routes`.  Everything but the path -- grids, limits, weights,
        radii, footprint -- stays this planner's.  plan() keeps planning on the constructor's path (route 0)."""
        spline_tables(reference_path)            # a path without numeric coefficients is refused here, on the host
        self.routes.append(reference_path)
        if self._engine is not None:
            rid = self._engine.add_route(reference_path)
            assert rid == len(self.routes) - 1, (rid, len(self.routes))
        return len(self.routes) - 1

    def resolve_limits(self, constraint_overrides) -> np.ndarray:
        """[max_speed, max_accel, max_curvature, max_lat_accel] after overrides (frenet_planner.py:921-930)."""
        lim = [self.max_speed, self.max_accel, self.max_curvature, self.max_lat_accel]
        if constraint_overrides:
            for i, key in enumerate(("max_speed", "max_accel", "max_curvature", "max_lat_accel")):
                lim[i] = constraint_overrides.get(key, lim[i])
        return np.array(lim, dtype=np.float64)

    # -- API -------------------------------------------------------------------------------
    def plan(self, ego_state, static_obstacles, dynamic_obstacles=None, target_speed: float = TARGET_SPEED,
             constraint_overrides: Optional[Dict[str, float]] = None, dynamic_obstacles_distribution=None,
             max_stop_distance: Optional[float] = None, _want_candidates: bool = False) -> Optional[FrenetPath]:
        """Best trajectory from the current ego state, or None (frenet_planner.py:227-304)."""
        self.last_check_stats = None
        self.last_result = None
        fs = self._cartesian_to_frenet_state(ego_state)
        if fs is None:
            return None
        return self.plan_from_frenet(fs.to_array(), static_obstacles, dynamic_obstacles, target_speed,
                                     constraint_overrides, dynamic_obstacles_distribution, max_stop_distance,
                                     _want_candidates)

    def plan_alternatives(self, ego_state, static_obstacles, dynamic_obstacles=None,
                          target_speed: float = TARGET_SPEED, constraint_overrides: Optional[Dict[str, float]] = None,
                          dynamic_obstacles_distribution=None, max_stop_distance: Optional[float] = None,
                          k: int = 5) -> List[FrenetPath]:
        """The k best feasible trajectories from the current ego state, best first (fewer when fewer are feasible):
        a fallback when the first choice is vetoed downstream.  Element 0 is what plan() returns, and the list is
        empty where plan() returns None.  Side effects are plan()'s: last_check_stats, the nearest-point cache and
        the curvature fed back from element 0.  Ranking: lower cost first, equal costs in generation order
        (include/fot.h, fot_ranked_t)."""
        if not 1 <= int(k) <= _lib.FOT_MAX_RANKED:
            raise ValueError(f"k must be in [1, {_lib.FOT_MAX_RANKED}]")
        self.last_check_stats = None
        self.last_result = None
        fs = self._cartesian_to_frenet_state(ego_state)
        if fs is None:
            return []
        res = self._sweep(fs.to_array(), static_obstacles, dynamic_obstacles, target_speed, constraint_overrides,
                          dynamic_obstacles_distribution, max_stop_distance, top_k=int(k))
        paths = [_frenet_path(a["series"], a["cost"]) for a in res.alternatives(0)]
        if paths:
            self._feed_back_curvature(paths[0])
        return paths

    def plan_under_weights(self, ego_state, static_obstacles, dynamic_obstacles=None,
                           target_speed: float = TARGET_SPEED, constraint_overrides: Optional[Dict[str, float]] = None,
                           dynamic_obstacles_distribution=None, max_stop_distance: Optional[float] = None,
                           weights=None) -> List[Optional[FrenetPath]]:
        """The trajectory a planner built with each weighting of the cost knobs would return from the current ego
        state, one entry per weighting (None where none is feasible under it), from ONE sweep.  `weights`: an
        [n_w, 6] array (columns _lib.COST_WEIGHT_KEYS) or a list of dicts keyed by those names, where a missing key
        takes this planner's own value.  Side effects are plan()'s, from this planner's own winner of the same
        launch: last_check_stats, the nearest-point cache and the curvature fed back.  Selection rule:
        include/fot.h, fot_weighted_t."""
        w = self.cost_weight_table(weights)
        self.last_check_stats = None
        self.last_result = None
        fs = self._cartesian_to_frenet_state(ego_state)
        if fs is None:
            return [None] * w.shape[0]
        res = self._sweep(fs.to_array(), static_obstacles, dynamic_obstacles, target_speed, constraint_overrides,
                          dynamic_obstacles_distribution, max_stop_distance, cost_weights=w)
        own = res.series(0)
        if own is not None:
            self._feed_back_curvature(_frenet_path(own, res.best_cost[0]))
        return [None if e is None else _frenet_path(e["series"], e["cost"]) for e in res.under_weights(0)]

    def assess(self, paths, static_obstacles, dynamic_obstacles=None, dynamic_obstacles_distribution=None,
               r2=None) -> Dict[str, np.ndarray]:
        """How close each of `paths` (FrenetPath objects: this planner's, plan_alternatives', or the reference
        planner's) comes to an obstacle field given as plan() takes it, on the device (fot_assess_trajectories,
        DESIGN.md section 4i).  Returns {name: array with one row per path} for the names of engine.ASSESS_FIELDS --
        dyn_min, dyn_at (n, circle, s, p), static_min, static_at (n, circle, point), and dyn_hits, first_hit,
        static_hit per threshold pair -- plus "collision_free" [m] bool under the planner's own pair.  r2: threshold
        pairs (r2_dyn, r2_static), one or [n_r, 2]; None: the planner's own pair for the field, under which
        collision_free is the verdict plan() gives the same positions (static_hit == 0 and dyn_hits <=
        floor(chance_epsilon * S)).  Only t, x, y and yaw of the paths are read."""
        import ctypes as C
        import torch
        series, lens = pack_paths(paths)
        user_r2 = None if r2 is None else assess_radii(r2)
        mode, dyn = classify_dynamic(dynamic_obstacles, dynamic_obstacles_distribution)
        static = None
        if static_obstacles is not None and len(static_obstacles) > 0:
            static = np.asarray(static_obstacles, dtype=np.float64).reshape(-1, 2)
        eng = self.engine
        own = eng.own_radii(mode)
        r2 = own if user_r2 is None else np.concatenate([own, user_r2])     # row 0: the verdict's own pair
        dev = torch.device("cuda", eng.device)
        t = {"series": torch.from_numpy(series).to(dev), "len": torch.from_numpy(lens).to(dev),
             "r2": torch.from_numpy(np.ascontiguousarray(r2)).to(dev)}
        b = _lib.FotBatch(n_q=1)
        if static is not None:
            t["static"] = torch.from_numpy(np.ascontiguousarray(static)).to(dev)
            b.static_obs, b.n_static = t["static"].data_ptr(), static.shape[0]
        if dyn is not None:
            t["dyn"] = torch.from_numpy(np.ascontiguousarray(dyn)).to(dev)
            b.dyn, b.dyn_mode = t["dyn"].data_ptr(), mode
            b.S, b.P, b.T_obs = dyn.shape[1], dyn.shape[2], dyn.shape[3]
        m, n_r = len(lens), r2.shape[0]
        a = _lib.FotAssessed(m=m, n_t=series.shape[-1], n_r=n_r, series=t["series"].data_ptr(), len=t["len"].data_ptr(),
                             r2=t["r2"].data_ptr())
        out = {}
        for name, dt, shape in ASSESS_FIELDS:
            out[name] = torch.empty((m, *(n_r if d == "r" else d for d in shape)), dtype=getattr(torch, dt), device=dev)
            setattr(a, name, out[name].data_ptr())
        eng.assess_device(b, a)                       # the handle's stream, synchronised
        res = {name: v.cpu().numpy() for name, v in out.items()}
        allowed = int(np.floor(self.chance_epsilon * b.S)) if mode == _lib.FOT_DYN_DISTRIBUTION else 0
        res["collision_free"] = (res["static_hit"][:, 0] == 0) & (res["dyn_hits"][:, 0] <= allowed)
        if user_r2 is not None:                       # the caller's pairs only
            for name in ("dyn_hits", "first_hit", "static_hit"):
                res[name] = res[name][:, 1:]
        return res

    def candidate_assessment(self, ego_state, static_obstacles, dynamic_obstacles=None,
                             target_speed: float = TARGET_SPEED, constraint_overrides: Optional[Dict[str, float]] = None,
                             dynamic_obstacles_distribution=None, max_stop_distance: Optional[float] = None,
                             assess_obstacles=None, r2=None) -> Optional[Dict[str, np.ndarray]]:
        """Every candidate plan() generates from the current ego state, the rejected ones included, with how close it
        comes to an obstacle field (fot_assess_candidates, DESIGN.md section 4j): {name: array with one row per
        candidate, in generation order} -- "cand_cat" (the sweep's category, _lib.CAT_*), "cand_cost", "keep" (samples
        assessed; 0 for an emptied candidate, whose row is blank: +inf, -1, 0) and the names of engine.ASSESS_FIELDS.
        The field is plan()'s own, or assess_obstacles [S, P, T, 2] (read as S samples, with plan()'s static points).
        r2: threshold pairs (r2_dyn, r2_static), one or [n_r, 2]; None: the planner's own pair for the field, under
        which a candidate of category OK, COLL or STOP is collision-free iff it is not COLL.  None where plan() returns
        None before sweeping (the ego state does not convert).  Side effects are plan()'s, from the winner of the same
        launch: last_check_stats, last_result, the nearest-point cache and the curvature fed back."""
        user_r2 = None if r2 is None else assess_radii(r2)               # checked before the device is used
        field = None
        if assess_obstacles is not None:
            field = np.asarray(assess_obstacles, dtype=np.float64)
            if field.ndim != 4 or field.shape[-1] != 2:
                raise ValueError(f"assess_obstacles must be [S, P, T, 2], got {list(field.shape)}")
            field = field[None]
        self.last_check_stats = None
        self.last_result = None
        fs = self._cartesian_to_frenet_state(ego_state)
        if fs is None:
            return None
        res = self._sweep(fs.to_array(), static_obstacles, dynamic_obstacles, target_speed, constraint_overrides,
                          dynamic_obstacles_distribution, max_stop_distance, want_candidates=True,
                          assess_candidates=True, assess_obstacles=field, assess_r2=user_r2)
        own = res.series(0)
        if own is not None:
            self._feed_back_curvature(_frenet_path(own, res.best_cost[0]))
        return res.candidate_assessment(0)

    def cost_weight_table(self, weights) -> np.ndarray:
        """[n_w, 6] float64 weightings (columns _lib.COST_WEIGHT_KEYS) from an [n_w, 6] array or a list of dicts keyed
        by those names; a key a dict leaves out takes this planner's own value.  Raises ValueError on anything else
        or on n_w outside [1, FOT_MAX_WEIGHT_SETS]."""
        keys = _lib.COST_WEIGHT_KEYS
        if isinstance(weights, dict):
            weights = [weights]
        if isinstance(weights, (list, tuple)) and weights and all(isinstance(d, dict) for d in weights):
            for d in weights:
                unknown = set(d) - set(keys)
                if unknown:
                    raise ValueError(f"unknown cost weight keys {sorted(unknown)}; expected a subset of {keys}")
            w = np.array([[float(d.get(k, getattr(self, k))) for k in keys] for d in weights], dtype=np.float64)
        else:
            w = np.asarray(weights, dtype=np.float64) if weights is not None else np.empty((0,))
            if w.ndim != 2 or w.shape[1] != len(keys):
                raise ValueError(f"weights must be [n_w, {len(keys)}] or a list of dicts keyed by {keys}")
        if not 1 <= w.shape[0] <= _lib.FOT_MAX_WEIGHT_SETS:
            raise ValueError(f"the number of weightings must be in [1, {_lib.FOT_MAX_WEIGHT_SETS}]")
        return w

    def plan_from_frenet(self, frenet_state, static_obstacles, dynamic_obstacles=None,
                         target_speed: float = TARGET_SPEED, constraint_overrides=None,
                         dynamic_obstacles_distribution=None, max_stop_distance=None,
                         _want_candidates: bool = False) -> Optional[FrenetPath]:
        """frenet_planner.py:271-304 for a given Frenet state [s, s_d, s_dd, d, d_d, d_dd]."""
        res = self._sweep(frenet_state, static_obstacles, dynamic_obstacles, target_speed, constraint_overrides,
                          dynamic_obstacles_distribution, max_stop_distance, want_candidates=_want_candidates)
        series = res.series(0)
        if series is None:
            return None
        return self._feed_back_curvature(_frenet_path(series, res.best_cost[0]))

    def _sweep(self, frenet_state, static_obstacles, dynamic_obstacles, target_speed, constraint_overrides,
               dynamic_obstacles_distribution, max_stop_distance, want_candidates: bool = False,
               top_k: int = 0, cost_weights=None, **assess) -> SweepResult:
        """One query through the sweep (ranked when top_k > 0, selected under each weighting of cost_weights [n_w, 6]
        when given); sets last_result and last_check_stats."""
        mode, dyn = classify_dynamic(dynamic_obstacles, dynamic_obstacles_distribution)
        static = None
        if static_obstacles is not None and len(static_obstacles) > 0:
            static = np.asarray(static_obstacles, dtype=np.float64).reshape(-1, 2)
        q = query_arrays(np.reshape(frenet_state, (1, 6)), float(target_speed), self.resolve_limits(constraint_overrides),
                         max_stop_distance, static, dyn, mode, self.d_t_s)
        res = self._run(q, want_candidates, top_k=top_k, cost_weights=cost_weights, **assess)
        self.last_result = res
        stats = {key: int(res.stats[0, _lib.STAT_KEYS.index(key)]) for key in _REF_STAT_ORDER}
        if max_stop_distance is not None:
            stats["stop_distance_error"] = int(res.stats[0, _lib.STAT_KEYS.index("stop_distance_error")])
        self.last_check_stats = stats
        return res

    def _run(self, q: QueryArrays, want_candidates: bool = False, winner_samples: int = 0, top_k: int = 0,
             rank_series: bool = True, cost_weights=None, weight_series: bool = True,
             cost_terms: bool = False, assess: bool = False, assess_obstacles=None, assess_r2=None,
             assess_candidates: bool = False) -> SweepResult:
        """Sweep the batch q: as a device-resident `DeviceBatch` when it asks for ranked alternatives, cost weightings,
        cost terms or an assessment (outputs only the device-side calls produce), otherwise through the host-pointer
        call."""
        if top_k > 0 or cost_weights is not None or cost_terms or assess or assess_candidates:
            from .batch import DeviceBatch           # batch.py builds on this module
            db = DeviceBatch(self, q.frenet, q.target, q.dyn, q.dyn_mode, limits=q.limits, max_stop_distance=q.stop,
                             static_obstacles=q.static, top_k=top_k, rank_series=rank_series,
                             cost_weights=cost_weights, weight_series=weight_series, cost_terms=cost_terms,
                             route=q.route, assess=assess, assess_obstacles=assess_obstacles, assess_r2=assess_r2,
                             assess_candidates=assess_candidates,
                             candidate_table=assess_candidates and want_candidates)
            db.launch()
            return db.sweep_result(want_candidates, winner_samples)
        return self.engine.run_host(q, want_candidates, winner_samples)

    def _feed_back_curvature(self, path: FrenetPath) -> FrenetPath:
        """The ego curvature the next call starts from (frenet_planner.py:301-302)."""
        if len(path.c) > 1:
            self._last_kappa = float(path.c[1])
        return path

    def reset_ego_curvature(self):
        """frenet_planner.py:326-332."""
        self._last_kappa = 0.0

    def _cartesian_to_frenet_state(self, ego_state) -> Optional[FrenetState]:
        """frenet_planner.py:334-374."""
        arr = ego_to_frenet(self.converter, ego_state, self._last_kappa)
        return None if arr is None else FrenetState(*arr)
