#!/usr/bin/env python
"""Generate the golden fixtures by running the UNMODIFIED reference planner.

Run in the build container only (it imports /root/reference read-only):

    python tests/golden/make_golden.py

Writes, next to this file:
  standard_queries.npz   for every tests.scenarios.standard_queries() case: the reference's Frenet
                         state, per-candidate category and cost, chosen index, last_check_stats and
                         the 15 winner sequences
  closed_loop_s01.npz    a subset of the plan() calls of a closed-loop run of scenarios/scenario_01_cv.yaml
                         (pysocialforce stubbed, pedestrians replayed at constant velocity, CV predictor;
                         SURVEY.md section 8c): inputs of each call and the reference's outputs
The reference holds no golden vectors of its own, so these files are what pins the oracle and the
CUDA path to the reference's behaviour on the GPU box, where /root/reference does not exist.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("FOT_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)      # our `tests` package must shadow the reference's
sys.modules.setdefault("pysocialforce", types.ModuleType("pysocialforce"))   # not installed; unused by the planner

from loguru import logger  # noqa: E402

logger.remove()

from src.core.data_structures import EgoVehicleState  # noqa: E402
from src.core.footprint import EgoFootprint  # noqa: E402
from src.planning.cubic_spline import CubicSpline2D  # noqa: E402
from src.planning.frenet_planner import FrenetPlanner  # noqa: E402

from tests import scenarios  # noqa: E402

CAT_NAMES = ("ok", "max_speed_error", "max_accel_error", "max_curvature_error", "max_lat_accel_error",
             "road_bound_error", "collision_error", "stop_distance_error")
CAT_DROP = 8
SERIES = ("t", "s", "s_d", "s_dd", "s_ddd", "d", "d_d", "d_dd", "d_ddd", "x", "y", "yaw", "c", "v", "a")


def reference_plan(planner, ego, static, dyn, target, overrides, dist, msd):
    """plan() through the reference's own steps (frenet_planner.py:261-304), keeping every
    candidate's category."""
    planner.last_check_stats = None
    fs = planner._cartesian_to_frenet_state(ego)
    if fs is None:
        return None
    fps = planner._generate_frenet_paths(fs, target)
    index = {id(fp): i for i, fp in enumerate(fps)}
    costs = np.array([fp.cost for fp in fps], dtype=np.float64)
    fps = planner._calc_global_paths(fps)
    groups = planner._check_paths(fps, static, dyn, overrides, dist)
    if msd is not None:
        planner._apply_stop_distance_filter(groups, msd)
    cats = np.full(len(fps), CAT_DROP, dtype=np.uint8)
    for name, members in groups.items():
        for fp in members:
            cats[index[id(fp)]] = CAT_NAMES.index(name)
    stats = {k: len(v) for k, v in groups.items()}
    planner.last_check_stats = stats
    best = planner._select_best_path(groups)
    if best is not None and len(best.c) > 1:
        planner._last_kappa = float(best.c[1])
    out = {"fs": np.array(fs.to_array(), dtype=np.float64), "cats": cats, "costs": costs,
           "best": np.int64(index[id(best)] if best is not None else -1),
           "stats": np.array([stats.get(k, -1) for k in CAT_NAMES], dtype=np.int64)}
    if best is not None:
        out["cost"] = np.float64(best.cost)
        for name in SERIES:
            out["w_" + name] = np.asarray(getattr(best, name), dtype=np.float64)
    return out


def make_standard():
    store = {}
    for q in scenarios.standard_queries():
        fp = None if q.footprint is None else EgoFootprint.multi_circle(*q.footprint)
        kw = dict(q.knobs)
        if fp is not None:
            kw["footprint"] = fp
        planner = FrenetPlanner(CubicSpline2D(*q.waypoints), **kw)
        planner._last_kappa = q.last_kappa
        static = np.empty((0, 2)) if q.static is None else q.static
        res = reference_plan(planner, EgoVehicleState(*q.ego), static, q.dyn, q.target_speed, q.overrides,
                             q.dist, q.max_stop_distance)
        for k, v in res.items():
            store[f"{q.name}/{k}"] = v
        print(f"{q.name}: {len(res['cats'])} candidates, best {int(res['best'])}")
    np.savez_compressed(os.path.join(HERE, "standard_queries.npz"), **store)


def make_closed_loop(max_calls=96):
    """Config 1: scenario_01_cv closed loop; the reference planner drives the simulation and every
    plan() call is recorded (a spread of up to `max_calls` of them is stored, always including the calls
    made with constraint overrides, i.e. the CAUTION / EMERGENCY retries)."""
    import yaml
    from src.config import SimulationConfig, validate_config
    from src.simulation.integrated_simulator import IntegratedSimulator
    from src.simulation.replay_source import ReplayPedestrianSource

    with open(os.path.join(REF, "scenarios", "scenario_01_cv.yaml")) as f:
        d = yaml.safe_load(f)
    peds = np.array(d.pop("ped_initial_states"), dtype=float)
    d.pop("ped_groups", None)
    d["sgan_model_path"] = None
    d["visualization_enabled"] = False
    d["prediction_method"] = "cv"
    cfg = SimulationConfig(**d)
    validate_config(cfg)
    sim = IntegratedSimulator(cfg)
    n_frames = int(cfg.total_time / cfg.dt) + 200
    t = np.arange(n_frames)[:, None, None] * cfg.dt
    traj = peds[None, :, 0:2] + peds[None, :, 2:4] * t
    sim.pedestrian_sim = ReplayPedestrianSource(traj, dt=cfg.dt)

    calls = []
    planner = sim.planner
    original = planner.plan

    def recording_plan(ego_state, static_obstacles, dynamic_obstacles=None, target_speed=None,
                       constraint_overrides=None, dynamic_obstacles_distribution=None, max_stop_distance=None):
        rec = {"ego": np.array([ego_state.x, ego_state.y, ego_state.yaw, ego_state.v, ego_state.a], dtype=np.float64),
               "last_kappa": np.float64(planner._last_kappa),
               "prev_s": np.float64(getattr(planner.converter, "_prev_s", np.nan)),
               "target": np.float64(target_speed),
               "dyn": np.array(dynamic_obstacles, dtype=np.float64),
               "ovr": np.array([np.nan if not constraint_overrides else constraint_overrides.get(k, np.nan)
                                for k in ("max_speed", "max_accel", "max_curvature", "max_lat_accel")]),
               "msd": np.float64(np.nan if max_stop_distance is None else max_stop_distance)}
        assert dynamic_obstacles_distribution is None
        assert static_obstacles is None or len(static_obstacles) == 0
        ovr = constraint_overrides
        res = reference_plan(planner, ego_state, static_obstacles, dynamic_obstacles, target_speed, ovr, None,
                             max_stop_distance)
        rec.update({"fs": res["fs"], "cats": res["cats"], "costs": res["costs"], "best": res["best"],
                    "stats": res["stats"]})
        if int(res["best"]) >= 0:
            rec["cost"] = res["cost"]
            for name in ("x", "y", "v", "c"):
                rec["w_" + name] = res["w_" + name]
        calls.append(rec)
        # hand the simulator the reference's own answer (planner state already advanced above)
        planner._last_kappa = float(rec["last_kappa"])
        if hasattr(planner.converter, "_prev_s") and not np.isnan(rec["prev_s"]):
            planner.converter._prev_s = float(rec["prev_s"])
        elif hasattr(planner.converter, "_prev_s"):
            del planner.converter._prev_s
        return original(ego_state, static_obstacles, dynamic_obstacles, target_speed, constraint_overrides,
                        dynamic_obstacles_distribution, max_stop_distance)

    planner.plan = recording_plan
    sim.warmup()
    sim.run()
    n = len(calls)
    forced = [i for i, c in enumerate(calls) if not np.all(np.isnan(c["ovr"]))]
    spread = list(np.linspace(0, n - 1, max(2, max_calls - min(len(forced), max_calls // 2))).astype(int))
    keep = sorted(set(forced[: max_calls // 2]) | set(spread))
    # every third kept call without overrides is left out, which keeps the file under 1 MB; every retry stays
    plain = [i for i in keep if i not in set(forced)]
    keep = sorted(set(keep) - set(plain[2::3]))
    store = {"n_calls_total": np.int64(n), "kept": np.array(keep, dtype=np.int64),
             "waypoints_x": np.array(cfg.reference_waypoints_x, dtype=np.float64),
             "waypoints_y": np.array(cfg.reference_waypoints_y, dtype=np.float64)}
    for j, i in enumerate(keep):
        for k, v in calls[i].items():
            store[f"c{j}/{k}"] = v
    np.savez_compressed(os.path.join(HERE, "closed_loop_s01.npz"), **store)
    states = {}
    for c in calls:
        key = "normal" if np.all(np.isnan(c["ovr"])) else ("emergency" if c["target"] == 0.0 else "caution")
        states[key] = states.get(key, 0) + 1
    print(f"closed loop: {n} plan() calls ({states}), stored {len(keep)}; steps {len(sim.history)}")


if __name__ == "__main__":
    make_standard()
    make_closed_loop()
    for f in ("standard_queries.npz", "closed_loop_s01.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")
