"""Batched closed-loop roll-out driver (SURVEY.md section 8f, rank 3).

The reference runs its campaigns (Monte-Carlo seeds, sensitivity sweeps: examples/run_da_poc.py:179+,
examples/run_rq1b_sensitivity.py:64, examples/run_statistical_benchmark.py:243-261) as sequential loops of
`IntegratedSimulator.step()`.  This driver advances N independent simulations in lock-step and issues ONE
batched sweep per (re)planning attempt:

    replayed pedestrians -> observer (0.4 s sampling) -> CV prediction + t = 0 column   [device]
                         -> safety metrics (clearance, clearance ahead)                  [device]
                         -> fail-safe state machine: target speed, limits, stop room     [host, vectorised]
                         -> FrenetPlanner sweep, up to 3 escalation retries per step     [device]
                         -> ego update from the winner's second sample, or the adaptive emergency stop

It restates, per simulation, exactly what `IntegratedSimulator.step()` / `run()` do with a replayed
pedestrian source and the constant-velocity predictor (src/simulation/integrated_simulator.py:406-422,
:424-527, :529-653, :655-676, :678-747, :749-802, :842-892; src/core/state_machine.py:116-278;
src/pedestrian/observer.py:52-86; src/simulation/replay_source.py:31-111), so that a batch reproduces the
reference's trajectories (tests/test_gpu_rollout.py, golden roll-outs recorded from the unmodified
reference by tests/golden/make_golden_rollout.py).  Pedestrian ground truth stays outside (replay), as in
the reference's own pysocialforce-free source; static obstacles and the ego footprint (single circle or the
multi-circle cover) are shared by the simulations of a batch.  The reference path may differ: with `routes`, each
simulation drives its own (DESIGN.md section 4h), so that a campaign over several scenarios' roads is one lock-step.
"""
from __future__ import annotations

import math
import time
from typing import Dict, Optional

import numpy as np

from . import _lib
from .batch import BatchFrenetPlanner, DeviceBatch
from .engine import route_array
from .frenet_host import BatchCoordinateConverter, RoutedCoordinateConverter, ego_to_frenet_many
from .prediction import DevicePredictionPostprocessor, safety_metrics
from .spline import CubicSpline2D

NORMAL, CAUTION, EMERGENCY = 0, 1, 2
SGAN_DT = 0.4          # the observer samples at the SGAN rate whatever the simulation dt (integrated_simulator.py:325)


def _knob(knobs, key, default):
    v = knobs.get(key, default)
    if v is None or (isinstance(v, float) and math.isnan(v)):
        return default
    return v


class _Footprint:
    """EgoFootprint.multi_circle (src/core/footprint.py:27-42): n equal circles along the heading axis covering the
    vehicle_length x vehicle_width rectangle."""

    def __init__(self, vehicle_length: float, vehicle_width: float, n_circles: int):
        if n_circles < 1:
            raise ValueError(f"n_circles must be >= 1, got {n_circles}")
        seg = vehicle_length / n_circles
        self.offsets = -vehicle_length / 2 + seg / 2 + seg * np.arange(n_circles)
        self.radius = float(np.hypot(seg / 2, vehicle_width / 2))


def footprint_from_knobs(k) -> Optional[_Footprint]:
    """footprint_from_config (footprint.py:68-78): None = the legacy single circle of ego_radius."""
    mode = k.get("ego_footprint", None)
    multi = mode == "multi_circle" or bool(k.get("ego_footprint_multi_circle", 0.0))
    if not multi:
        return None
    return _Footprint(_knob(k, "vehicle_length", 4.5), _knob(k, "vehicle_width", 2.0), int(_knob(k, "ego_footprint_n_circles", 3)))


def expand_static_obstacles(static_obstacles, step: float = 0.5) -> np.ndarray:
    """Boundary points of rectangular obstacles for the planner's point-obstacle test
    (integrated_simulator.py:804-836: edges sampled every `step`, duplicates removed, rows sorted by np.unique).
    An [M, 2] array is taken as points already."""
    if static_obstacles is None or len(static_obstacles) == 0:
        return np.empty((0, 2))
    arr = np.asarray(static_obstacles, dtype=np.float64)
    if arr.ndim == 2 and arr.shape[1] == 2:
        return np.ascontiguousarray(arr)
    pts = []
    for rect in static_obstacles:
        if len(rect) != 4:
            continue
        x_min, x_max, y_min, y_max = rect
        xs = np.arange(x_min, x_max + step, step)
        ys = np.arange(y_min, y_max + step, step)
        for x in xs:
            pts.append((x, y_min))
            pts.append((x, y_max))
        for y in ys:
            pts.append((x_min, y))
            pts.append((x_max, y))
    if not pts:
        return np.empty((0, 2))
    return np.unique(np.array(pts), axis=0)


class _StateMachines:
    """FailSafeStateMachine for N simulations at once (src/core/state_machine.py:29-278)."""

    def __init__(self, n: int, k: Dict[str, float]):
        self.k = k
        self.state = np.zeros(n, dtype=np.int64)
        self.failures = np.zeros(n, dtype=np.int64)
        fp = footprint_from_knobs(k)                                                               # effective_ego_radius
        combined = (fp.radius if fp is not None else _knob(k, "ego_radius", 1.0)) + _knob(k, "ped_radius", 0.2)   # :44-46
        rc, re = k.get("state_machine_recover_clearance_caution"), k.get("state_machine_recover_clearance_emergency")
        nan = lambda v: v is None or (isinstance(v, float) and math.isnan(v))
        self.clearance_caution = _knob(k, "state_machine_safe_distance_caution", 2.0) - combined if nan(rc) else rc
        self.clearance_emergency = _knob(k, "state_machine_safe_distance_emergency", 3.0) - combined if nan(re) else re
        self.trigger_clearance = _knob(k, "state_machine_trigger_clearance_caution", 0.0)
        self.trigger_headway = _knob(k, "state_machine_trigger_time_headway", 0.0)
        self.envelope_decel = _knob(k, "state_machine_envelope_decel", 0.0)
        self.envelope_standoff = _knob(k, "state_machine_envelope_standoff", 0.5)
        self.last_clearance = np.full(n, np.inf)
        self.last_clearance_ahead = np.full(n, np.inf)

    def update(self, idx, found, clearance, clearance_ahead, ego_speed):
        """state_machine.py:116-179 for the simulations `idx` (array form of the per-state branches)."""
        idx = np.asarray(idx, dtype=np.int64)
        ok = np.asarray(found, dtype=bool)
        cl = np.asarray(clearance, dtype=np.float64)
        self.last_clearance[idx] = cl
        self.last_clearance_ahead[idx] = clearance_ahead
        trig = self.trigger_clearance + self.trigger_headway * np.maximum(np.asarray(ego_speed, dtype=np.float64), 0.0)
        st, fails = self.state[idx], self.failures[idx]
        new_st, new_f = st.copy(), fails.copy()
        normal, caution, emergency = st == NORMAL, st == CAUTION, st == EMERGENCY
        # NORMAL: failure -> CAUTION (+1); preventive trigger -> CAUTION (counter 0); else counter 0
        m = normal & ~ok
        new_st[m], new_f[m] = CAUTION, fails[m] + 1
        m = normal & ok & (trig > 0.0) & (cl < trig)
        new_st[m], new_f[m] = CAUTION, 0
        m = normal & ok & ~((trig > 0.0) & (cl < trig))
        new_f[m] = 0
        # CAUTION: clean success -> NORMAL when the clearance gate is open; failure -> EMERGENCY (+1); else counter 0
        m = caution & ok & (fails == 0) & (cl > np.maximum(self.clearance_caution, trig))
        new_st[m] = NORMAL
        m = caution & ~ok
        new_st[m], new_f[m] = EMERGENCY, fails[m] + 1
        m = caution & ok & (fails != 0)
        new_f[m] = 0
        # EMERGENCY: success with a wide clearance -> CAUTION
        m = emergency & ok & (cl > self.clearance_emergency)
        new_st[m] = CAUTION
        self.state[idx], self.failures[idx] = new_st, new_f

    def planner_config(self, idx):
        """state_machine.py:181-278: (target speed, limits [n,4], max_stop_distance (NaN = none))."""
        k = self.k
        idx = np.asarray(idx, dtype=np.int64)
        n = len(idx)
        v_target = float(k["ego_target_speed"])
        lat = _knob(k, "ego_max_lat_accel", 3.0)
        limits = np.tile(np.array([k["ego_max_speed"], k["ego_max_accel"], k["ego_max_curvature"], lat], dtype=np.float64), (n, 1))
        ca = self.last_clearance_ahead[idx]
        seen = np.isfinite(ca)
        with np.errstate(invalid="ignore"):
            # safe-speed envelope (:252-266) and stop room (:268-278); NaN = None
            env_on = (self.envelope_decel > 0.0) & seen
            v_env = np.where(env_on, np.sqrt(2.0 * self.envelope_decel * np.maximum(np.where(seen, ca, 0.0) - self.envelope_standoff, 0.0)), np.nan)
            room = np.where(seen, np.maximum(np.where(seen, ca, 0.0) - 0.2, 0.05), np.nan)
        st = self.state[idx]
        normal, caution, emergency = st == NORMAL, st == CAUTION, st == EMERGENCY
        target = np.full(n, v_target)
        msd = np.full(n, np.nan)
        m = normal & env_on & (v_env < v_target)
        target[m] = v_env[m]
        speed_mult = _knob(k, "state_machine_caution_speed_multiplier", 0.8)
        t_c = np.where(env_on, np.minimum(v_target * speed_mult, np.where(env_on, v_env, 0.0)), v_target * speed_mult)
        target[caution] = t_c[caution]
        m = caution & env_on & (v_env <= 0.0)
        msd[m] = room[m]
        limits[caution, 1] = k["ego_max_accel"] * _knob(k, "state_machine_caution_accel_multiplier", 1.5)
        limits[caution, 0] = k["ego_max_speed"] * speed_mult
        target[emergency] = 0.0
        limits[emergency, 1] = k["ego_max_accel"] * _knob(k, "state_machine_emergency_accel_multiplier", 3.0)
        limits[emergency, 3] = lat * _knob(k, "state_machine_emergency_lat_accel_multiplier", 2.0)
        if self.envelope_decel > 0.0:
            m = emergency & seen
            msd[m] = room[m]
        return target, limits, msd


class BatchedClosedLoop:
    """N closed-loop simulations of the reference's planning stack, advanced in lock-step.

    waypoints_x / waypoints_y : the reference path (route 0)
    routes       : [(wx, wy), ...] further reference paths, routes 1, 2, ...; None: none
    route        : [N] route of each simulation (an integer for all; None: route 0).  Planning, the nearest-point
                   caches and the goal check (`s[-1] - s_now < 2.0`) follow each simulation's own path; a simulation
                   gives what a loop over its path alone gives.
    knobs        : SimulationConfig fields by name (dt, obs_len, ego_*, planner and state-machine knobs)
    ped_tracks   : [N, T_frames, P, 2] replayed pedestrian positions, one frame per dt
    ego0         : [N, 5] initial (x, y, yaw, v, a)
    sampler      : None = the constant-velocity predictor.  Otherwise the stand-in for the reference's trajectory
                   generator (SGAN; outside the hot path): `sampler(obs [n, obs_len, P, 2], idx) -> raw [n, S, pred_len,
                   P, 2]`, the generator's absolute predictions at the 0.4 s cadence for the active simulations `idx`,
                   S = knobs["num_samples"].  Everything after the generator runs on the device: resampling onto the
                   planner grid, closest-to-mean selection, t = 0 column (trajectory_predictor.py:233-353,
                   integrated_simulator.py:503-525).  With knobs["distribution_aware_planning"] the planner sweeps
                   against the whole sample set under the chance constraint knobs["chance_epsilon"]
                   (integrated_simulator.py:457-460, :582; frenet_planner.py:1076-1124), else against the
                   representative sample.
    assess       : also assess every step's executed plan (fot_assess_trajectories, DESIGN.md section 4i) against the
                   whole sample set with its t = 0 column when there is a sampler -- even when planning used the
                   representative sample -- else against the tensor planned against, under the planner's own radius
                   pair; run() then also returns plan_min_distance (closest approach to any predicted sample) and
                   plan_hit_fraction (dyn_hits / S: the share of the S samples the plan collides with), [N, steps],
                   NaN where no plan was executed (none found, or a winner of fewer than 2 samples, which the ego
                   does not follow).  Nothing else changes.
    """

    def __init__(self, waypoints_x, waypoints_y, knobs: Dict[str, float], ped_tracks: np.ndarray, ego0: np.ndarray,
                 device: int = 0, static_obstacles=None, record: bool = False, sampler=None, cost_weights=None,
                 routes=None, route=None, assess: bool = False):
        k = {key: (None if (isinstance(v, float) and math.isnan(v)) else v) for key, v in knobs.items()}
        self.k = k
        self.dt = float(k["dt"])
        # static obstacles, shared by all simulations: boundary points [M, 2], or rectangles
        # [x_min, x_max, y_min, y_max] expanded as IntegratedSimulator._expand_static_obstacles does
        self.static_points = expand_static_obstacles(static_obstacles)
        self.tracks = np.ascontiguousarray(ped_tracks, dtype=np.float64)
        self.n, self.n_frames, self.P, _ = self.tracks.shape
        self.ego = np.array(ego0, dtype=np.float64).reshape(self.n, 5).copy()
        self.spline = CubicSpline2D(list(waypoints_x), list(waypoints_y))
        self.paths = [self.spline] + [CubicSpline2D(list(wx), list(wy)) for wx, wy in (routes or [])]
        self.route = route_array(route, self.n, len(self.paths))            # None: every simulation on route 0
        self.ego_radius, self.ped_radius = _knob(k, "ego_radius", 1.0), _knob(k, "ped_radius", 0.3)
        self.footprint = footprint_from_knobs(k)
        self.planner = BatchFrenetPlanner(
            self.spline, max_speed=k["ego_max_speed"], max_accel=k["ego_max_accel"], max_curvature=k["ego_max_curvature"],
            max_lat_accel=_knob(k, "ego_max_lat_accel", 3.0), dt=self.dt, d_road_w=k["d_road_w"],
            max_road_width=k["max_road_width"], robot_radius=self.ego_radius,
            obstacle_radius=_knob(k, "obstacle_radius", self.ped_radius), min_t=_knob(k, "min_t", 4.0),
            max_t=_knob(k, "max_t", 5.0), d_t_s=_knob(k, "d_t_s", 5.0 / 3.6), k_j=k["k_j"], k_t=k["k_t"], k_d=k["k_d"],
            k_s_dot=k["k_s_dot"], k_lat=k["k_lat"], k_lon=k["k_lon"], chance_epsilon=_knob(k, "chance_epsilon", 0.0),
            collision_margin_inflation=_knob(k, "collision_margin_inflation", 1.0), footprint=self.footprint, device=device)
        for path in self.paths[1:]:
            self.planner.add_route(path)
        self.device = device
        # [N, 6] weighting of each simulation's cost (columns _lib.COST_WEIGHT_KEYS): every planning attempt selects
        # under it from the same sweep (fot_select_weighted) instead of under the knobs above; None: the knobs
        self.cost_weights = None
        if cost_weights is not None:
            self.cost_weights = np.ascontiguousarray(cost_weights, dtype=np.float64)
            if self.cost_weights.shape != (self.n, len(_lib.COST_WEIGHT_KEYS)):
                raise ValueError(f"cost_weights must be [{self.n}, {len(_lib.COST_WEIGHT_KEYS)}], "
                                 f"got {list(self.cost_weights.shape)}")
        self.assess = bool(assess)
        if self.assess and self.cost_weights is not None:
            raise ValueError("assess=True assesses the planner's own winner; it does not take cost_weights")
        self.last_assessment = None                     # (plan_min_distance, plan_hit_fraction) of the last step's idx
        self.post = DevicePredictionPostprocessor(pred_len=int(_knob(k, "pred_len", 12)), sgan_dt=SGAN_DT, sim_dt=self.dt,
                                                  plan_horizon=_knob(k, "max_t", 5.0), device=device)
        self.sampler = sampler
        self.num_samples = int(_knob(k, "num_samples", 1))
        self.distribution_aware = bool(_knob(k, "distribution_aware_planning", 0)) and self.num_samples >= 2 and sampler is not None
        self.fsm = _StateMachines(self.n, k)
        # per-simulation planner state: ego curvature cache and the two nearest-point caches (the planner's
        # converter and the simulator's own goal-check converter are separate objects in the reference)
        self.last_kappa = np.zeros(self.n)
        if self.route is None:
            self.plan_conv = BatchCoordinateConverter(self.spline, self.n, engine=self.planner.engine)
            self.goal_conv = BatchCoordinateConverter(self.spline, self.n, engine=self.planner.engine)
            self.path_end = None
        else:
            self.plan_conv = RoutedCoordinateConverter(self.paths, self.route, engine=self.planner.engine)
            self.goal_conv = RoutedCoordinateConverter(self.paths, self.route, engine=self.planner.engine)
            self.path_end = np.array([p.s[-1] for p in self.paths], dtype=np.float64)[self.route]   # s[-1] of each simulation's path
        # replayed pedestrians (replay_source.py:31-111): forward-difference velocities, shared clock
        vel = np.zeros_like(self.tracks)
        if self.n_frames >= 2:
            vel[:, :-1] = (self.tracks[:, 1:] - self.tracks[:, :-1]) / self.dt
            vel[:, -1] = vel[:, -2]
        self.vel = vel
        self.frame, self.ped_time = 0, 0.0
        # observer (observer.py:26-86), identical timing for every simulation
        self.obs_len = int(k["obs_len"])
        self.hist, self.hist_t, self.obs_acc, self.obs_last_t = [], [], 0.0, None
        self.time = 0.0
        self.active = np.ones(self.n, dtype=bool)
        self.reason = np.array(["timeout"] * self.n, dtype=object)
        self.n_plan_calls = 0
        # record=True keeps what IntegratedSimulator.save_results writes (full planned paths, predictions, metrics)
        self.record = bool(record)
        self.history = [[] for _ in range(self.n)]
        self.timers = {"frenet_host": 0.0, "sweep": 0.0, "prediction": 0.0, "metrics": 0.0, "total": 0.0}

    # -- pedestrians + observer -----------------------------------------------------------------
    def _ped_step(self):
        if self.frame < self.n_frames - 1:
            self.frame += 1
        self.ped_time += self.dt
        delta = self.dt if self.obs_last_t is None else max(self.ped_time - self.obs_last_t, 0.0)   # observer.py:58-66
        self.obs_last_t = self.ped_time
        self.obs_acc += delta
        if self.obs_acc + 1e-9 >= SGAN_DT:
            self.hist.append(self.tracks[:, self.frame].copy())
            self.hist_t.append(self.ped_time)
            self.hist, self.hist_t = self.hist[-self.obs_len:], self.hist_t[-self.obs_len:]
            self.obs_acc = max(self.obs_acc - SGAN_DT, 0.0)

    def warmup(self):
        """integrated_simulator.py:406-422."""
        for _ in range(int(self.obs_len * SGAN_DT / self.dt)):
            self._ped_step()

    # -- one planning attempt for the simulations `idx` -------------------------------------------
    def _plan(self, idx, target, limits, msd, dyn_dev, mode=_lib.FOT_DYN_SINGLE, assess_dev=None):
        import torch
        t0 = time.perf_counter()
        # ok False = conversion failure: plan() returns None (frenet_planner.py:346-374)
        frenet, ok = ego_to_frenet_many(self.plan_conv, idx, self.ego[idx], self.last_kappa[idx])
        self.n_plan_calls += len(idx)
        t1 = time.perf_counter()
        sel = torch.as_tensor(np.asarray(idx), device=dyn_dev.device)
        weights = None if self.cost_weights is None else self.cost_weights[np.asarray(idx)][:, None, :]
        batch = DeviceBatch(self.planner, frenet, target, dyn_dev.index_select(0, sel), mode,
                            limits=limits, max_stop_distance=msd,
                            static_obstacles=self.static_points if len(self.static_points) else None,
                            cost_weights=weights, route=None if self.route is None else self.route[np.asarray(idx)],
                            assess=self.assess, assess_obstacles=None if assess_dev is None else assess_dev.index_select(0, sel))
        batch.launch(None)
        if weights is None:
            o_idx, o_len, o_cost, o_win = (batch.out[key] for key in ("best_idx", "winner_len", "best_cost", "winner"))
        else:                                                          # the winner under each simulation's weighting
            o_idx, o_len, o_cost, o_win = (batch.out[key][:, 0] for key in ("w_idx", "w_len", "w_cost", "w_series"))
        best = o_idx.cpu().numpy()
        wlen = o_len.cpu().numpy()
        win = o_win[:, 9:15, :2].cpu().numpy()                         # x y yaw c v a, first two samples
        found = ok & (best >= 0)
        if self.assess:                                                # the winner's closest approach and hit share
            S = (dyn_dev if assess_dev is None else assess_dev).shape[1]
            a_min = batch.out["a_dyn_min"][:, 0].cpu().numpy()
            a_frac = batch.out["a_dyn_hits"][:, 0, 0].cpu().numpy() / S
            self._last_assess = (np.where(found, a_min, np.nan), np.where(found, a_frac, np.nan))
        self._last_full = (o_win.cpu().numpy(), o_cost.cpu().numpy()) if self.record else None
        self.timers["frenet_host"] += t1 - t0
        self.timers["sweep"] += time.perf_counter() - t1
        return found, wlen, win

    # -- one simulation step for every active simulation -------------------------------------------
    def step(self):
        k, dt = self.k, self.dt
        t_step = time.perf_counter()
        idx = np.nonzero(self.active)[0]
        self._ped_step()
        pos, vel = self.tracks[:, self.frame], self.vel[:, self.frame]
        ts = self.ped_time
        # prediction (integrated_simulator.py:424-527): CV from the observer's last two float32 samples, or the
        # current positions alone while the observer is still filling
        ready = len(self.hist) >= self.obs_len
        mode, dist_dense, best_dense, assess_dev = _lib.FOT_DYN_SINGLE, None, None, None
        if ready and self.sampler is not None:
            # sample sets from the generator stand-in; everything behind it on the device
            import torch
            stale = max(ts - self.hist_t[-1], 0.0)
            obs = np.stack(self.hist, axis=1)                                  # [N, obs_len, P, 2]
            raw = np.asarray(self.sampler(obs[idx], idx), dtype=np.float64)    # [n, S, pred_len, P, 2]
            if raw.shape[0] != len(idx) or raw.shape[1] != self.num_samples:
                raise ValueError(f"sampler returned {raw.shape}, expected [{len(idx)}, {self.num_samples}, pred_len, P, 2]")
            full = np.zeros((self.n,) + raw.shape[1:])
            full[idx] = raw
            anchor = self.hist[-1].astype(np.float32).astype(np.float64)       # obs_traj[-1] is a float32 tensor (observer.py:131)
            if self.num_samples == 1:                                          # predict_single_best :336-338
                dense = self.post.process_prediction(full, anchor, stale)
                dyn = self.post.prepend_current(dense, pos, pick=torch.zeros(self.n, dtype=torch.int32, device=dense.device), conditional=True)
                best_dense = dense[:, 0]
            else:
                dense = self.post.process_prediction(full, anchor, stale)
                best, _ = self.post.select_best(dense)
                dyn = self.post.prepend_current(dense, pos, pick=best, conditional=True)
                best_dense = dense[torch.arange(self.n, device=dense.device), best.long()]
                dist_dense = dense
                if self.distribution_aware:
                    dyn = self.post.prepend_current(dense, pos, pick=None, conditional=False)
                    mode = _lib.FOT_DYN_DISTRIBUTION
                elif self.assess:                                      # the whole sample set, t = 0 column included
                    assess_dev = self.post.prepend_current(dense, pos, pick=None, conditional=False)
        elif ready:
            stale = max(ts - self.hist_t[-1], 0.0)
            dyn = self.post.predict_cv(self.hist[-1], self.hist[-2], stale, pos, obs_float32=True)
        else:
            import torch
            dyn = torch.from_numpy(np.ascontiguousarray(pos[:, None, :, None, :])).to(self.post._dev)
        rec = None
        if self.record:
            if ready and self.sampler is not None:
                pred = best_dense.cpu().numpy()
                dist = dist_dense.cpu().numpy() if dist_dense is not None else None
            else:
                pred = self.post.predict_cv(self.hist[-1], self.hist[-2], stale, None, obs_float32=True)[:, 0].cpu().numpy() if ready else None
                dist = None
            rec = {"time": self.time, "pred": pred, "dist": dist, "old_a": self.ego[:, 4].copy()}
        t_pred = time.perf_counter()
        m = safety_metrics(self.ego, pos, vel, self.ego_radius, self.ped_radius, footprint=self.footprint, device=self.device)
        clearance, ahead = m["clearance"].cpu().numpy(), m["clearance_ahead"].cpu().numpy()
        self.timers["prediction"] += t_pred - t_step
        self.timers["metrics"] += time.perf_counter() - t_pred
        last_clearance = ahead.copy()                                  # :566-567 feeds the emergency stop

        # planning cycle with escalation retries (:529-653)
        state_before = self.fsm.state[idx].copy()
        target, limits, msd = self.fsm.planner_config(idx)
        found, wlen, win = self._plan(idx, target, limits, msd, dyn, mode, assess_dev)
        if self.assess:
            a_min, a_frac = self._last_assess
        if self.record:
            full_w, full_c = (a.copy() for a in self._last_full)
        self.fsm.update(idx, found, clearance[idx], ahead[idx], self.ego[idx, 3])
        attempts = np.zeros(len(idx), dtype=np.int64)
        calls = np.ones(len(idx), dtype=np.int64)
        while True:
            retry = np.nonzero(~found & (self.fsm.state[idx] != state_before) & (attempts < 3))[0]
            if len(retry) == 0:
                break
            attempts[retry] += 1
            calls[retry] += 1
            sub = idx[retry]
            t2, l2, m2 = self.fsm.planner_config(sub)
            f2, w2, win2 = self._plan(sub, t2, l2, m2, dyn, mode, assess_dev)
            found[retry], wlen[retry], win[retry] = f2, w2, win2
            if self.assess:
                a_min[retry], a_frac[retry] = self._last_assess
            if self.record:
                full_w[retry], full_c[retry] = self._last_full
            failed = retry[~f2]
            state_before[failed] = self.fsm.state[idx[failed]]
            if len(failed):
                self.fsm.update(idx[failed], np.zeros(len(failed), bool), clearance[idx[failed]], ahead[idx[failed]],
                                self.ego[idx[failed], 3])

        # ego update (:655-676) or adaptive emergency stop (:749-802)
        follow = found & (wlen >= 2)
        if self.assess:                                                # a winner shorter than 2 samples is not executed
            a_min[~follow], a_frac[~follow] = np.nan, np.nan
        f_idx = idx[follow]
        self.ego[f_idx] = win[follow][:, [0, 1, 2, 4, 5], 1]          # x y yaw v a of the winner's second sample
        self.last_kappa[f_idx] = win[follow][:, 3, 1]                  # frenet_planner.py:301-302
        for i in idx[~follow]:                                         # the few without a path: scalar, as the reference computes it
            cap = k.get("ego_emergency_decel") or k["ego_max_accel"] * 2.0
            cl = float(last_clearance[i])
            x, y, yaw, v, a = self.ego[i]
            required = v ** 2 / (2.0 * max(cl - 0.2, 0.05)) if math.isfinite(cl) else cap
            max_dec = float(np.clip(required, k["ego_max_accel"], cap))
            x += v * np.cos(yaw) * dt
            y += v * np.sin(yaw) * dt
            v = max(0.0, v - max_dec * dt)
            self.ego[i] = [x, y, yaw, v, -max_dec if v > 0 else 0.0]
            self.last_kappa[i] = 0.0                                   # planner.reset_ego_curvature()
        # termination (:870-886): collision of the NEW ego state with the same pedestrian frame, then the goal
        t_m = time.perf_counter()
        m2 = safety_metrics(self.ego, pos, vel, self.ego_radius, self.ped_radius, footprint=self.footprint, device=self.device)
        collided = m2["collision"].cpu().numpy()
        self.timers["metrics"] += time.perf_counter() - t_m
        hit = idx[collided[idx]]
        self.active[hit], self.reason[hit] = False, "collision"
        alive = idx[~collided[idx]]
        if len(alive):
            s_now = self.goal_conv.nearest_s(alive, self.ego[alive, 0], self.ego[alive, 1])
            end = self.spline.s[-1] if self.path_end is None else self.path_end[alive]
            done = alive[end - s_now < 2.0]
            self.active[done], self.reason[done] = False, "goal"
        if self.record:
            md, ttc = m2["min_distance"].cpu().numpy(), m2["ttc"].cpu().numpy()
            names = ("NORMAL", "CAUTION", "EMERGENCY")
            for j, i in enumerate(idx):
                n_w = int(wlen[j]) if found[j] else 0
                self.history[i].append({
                    "time": rec["time"], "ego": self.ego[i].copy(), "jerk": (self.ego[i, 4] - rec["old_a"][i]) / dt,
                    "state": names[int(self.fsm.state[i])], "min_distance": float(md[i]), "ttc": float(ttc[i]),
                    "collision": bool(collided[i]), "n_samples": self.num_samples,
                    "dist": None if rec["dist"] is None else rec["dist"][i],
                    "ped_pos": pos[i].copy(), "ped_vel": vel[i].copy(), "pred": None if rec["pred"] is None else rec["pred"][i],
                    "path": full_w[j][:, :n_w].copy() if found[j] else None, "cost": float(full_c[j]) if found[j] else float("inf")})
        if self.assess:
            self.last_assessment = (a_min, a_frac)
        self.time += dt
        self.timers["total"] += time.perf_counter() - t_step
        return idx, found, calls

    def save_results(self, i: int, output_dir: str, context: Optional[dict] = None) -> str:
        """The result files of simulation `i` as IntegratedSimulator.save_results writes them
        (integrated_simulator.py:894-1065): trajectory.npz with the same keys, shapes and construction,
        metrics_summary.csv and metrics_report.txt (results.py: the aggregate metrics of src/core/metrics.py and the
        context block; the four wall-clock entries avg/max_prediction/planning_time hold this driver's per-step
        times divided by the batch size).  Needs record=True.  `context` overrides entries of the context block
        (prediction_method, sgan_model, scenario_file, seed)."""
        import os
        from .results import aggregate_metrics, write_metrics_files
        if not self.record:
            raise RuntimeError("BatchedClosedLoop(record=True) is needed to write result files")
        h = self.history[i]
        os.makedirs(output_dir, exist_ok=True)
        col = lambda row: 9 + ("x", "y", "yaw", "c", "v", "a").index(row)         # winner block rows (types.SERIES)
        planned = lambda row: [np.array(r["path"][col(row)]) if r["path"] is not None else np.array([]) for r in h]
        goals = self.tracks[i, -1]
        path = os.path.join(output_dir, "trajectory.npz")
        np.savez(
            path,
            times=np.array([r["time"] for r in h]),
            ego_x=np.array([r["ego"][0] for r in h]), ego_y=np.array([r["ego"][1] for r in h]),
            ego_v=np.array([r["ego"][3] for r in h]), ego_yaw=np.array([r["ego"][2] for r in h]),
            ego_jerk=np.array([r["jerk"] for r in h]),
            ego_state=np.array([r["state"] for r in h]),
            min_distances=np.array([r["min_distance"] for r in h]), ttc=np.array([r["ttc"] for r in h]),
            proc_prediction=np.zeros(len(h)), proc_planning=np.zeros(len(h)),      # wall-clock per step: not reproduced
            ped_positions=np.array([r["ped_pos"] for r in h], dtype=object),
            ped_velocities=np.array([r["ped_vel"] for r in h], dtype=object),
            ped_goals=np.array([goals.copy() for _ in h], dtype=object),
            predicted_trajectories=np.array([r["pred"] if r["pred"] is not None else np.empty((0,)) for r in h], dtype=object),
            planned_x=np.array(planned("x"), dtype=object), planned_y=np.array(planned("y"), dtype=object),
            planned_v=np.array(planned("v"), dtype=object), planned_a=np.array(planned("a"), dtype=object),
            planned_yaw=np.array(planned("yaw"), dtype=object),
            planned_cost=np.array([r["cost"] for r in h]))
        metrics = aggregate_metrics(h, self.dt, prediction_dt=SGAN_DT, prediction_steps=int(_knob(self.k, "pred_len", 12)))
        steps_run = max(1, len(h))
        per_sim = 1.0 / (self.n * steps_run)
        metrics["avg_prediction_time"] = metrics["max_prediction_time"] = self.timers["prediction"] * per_sim
        metrics["avg_planning_time"] = metrics["max_planning_time"] = (self.timers["frenet_host"] + self.timers["sweep"]) * per_sim
        ctx = {"prediction_method": "cv" if self.sampler is None else "sgan", "sgan_model": None,
               "ego_target_speed": self.k["ego_target_speed"], "scenario_file": str(None), "seed": "not_set",   # :1013 str(getattr(config, 'config_path', ...))
               "termination_reason": str(self.reason[i]), "total_time": h[-1]["time"] + self.dt if h else 0.0,
               "steps": len(h)}
        if context:
            ctx.update(context)
        write_metrics_files(output_dir, ctx, metrics, any(r["collision"] for r in h))
        return path

    def run(self, n_steps: Optional[int] = None):
        """IntegratedSimulator.run (:842-892) for every simulation; returns per-simulation histories (with assess=True
        also plan_min_distance and plan_hit_fraction)."""
        if n_steps is None:
            n_steps = int(self.k["total_time"] / self.dt)
        ego_hist = np.full((self.n, n_steps, 5), np.nan)
        fsm_hist = np.full((self.n, n_steps), -1, dtype=np.int64)
        found_hist = np.zeros((self.n, n_steps), dtype=bool)
        calls_hist = np.zeros((self.n, n_steps), dtype=np.int64)
        steps = np.zeros(self.n, dtype=np.int64)
        if self.assess:
            min_hist, frac_hist = np.full((self.n, n_steps), np.nan), np.full((self.n, n_steps), np.nan)
        for s in range(n_steps):
            if not self.active.any():
                break
            idx, found, calls = self.step()
            ego_hist[idx, s] = self.ego[idx]
            fsm_hist[idx, s] = self.fsm.state[idx]
            found_hist[idx, s] = found
            calls_hist[idx, s] = calls
            steps[idx] += 1
            if self.assess:
                min_hist[idx, s], frac_hist[idx, s] = self.last_assessment
        out = {"ego": ego_hist, "fsm": fsm_hist, "found": found_hist, "calls": calls_hist, "steps": steps,
               "reason": self.reason.copy()}
        if self.assess:
            out["plan_min_distance"], out["plan_hit_fraction"] = min_hist, frac_hist
        return out
