"""Secondary measurements for BASELINE.json's configs 2, 3 and 5 (bench.py carries config 4).

  config 2  single plan() call, default grid, 50 pedestrians x 1 sample: p50 latency through the
            drop-in FrenetPlanner.plan() (host -> device -> host, FrenetPath rebuilt), time.perf_counter
            around the call exactly as the reference's simulator measures it
  config 3  dense grid 65 d x 32 T x 32 v vs 200 pedestrians x 20 samples, one call: kernel time
  config 5  state-machine relaxation: NORMAL / CAUTION / EMERGENCY plan() triple per step, 500 steps
Writes one JSON object to stdout.  GPU only; nothing here touches the oracle.
"""
import json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from tests import runners, scenarios
from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D, FrenetPlanner

out = {}
k = scenarios.S1_KNOBS

# ---- config 2 ---------------------------------------------------------------------------------
pl = FrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **k)
dyn = scenarios.pedestrian_field(np.random.default_rng(0), 50)
ego = runners._Ego(5.0, 0.0, 0.0, 5.0, 0.0)
static = np.empty((0, 2))
lat, kms = [], []
for i in range(103):
    pl.reset_ego_curvature()
    t0 = time.perf_counter()
    path = pl.plan(ego, static, dyn, 6.0)
    lat.append(time.perf_counter() - t0)
    kms.append(pl.last_result.kernel_ms)
lat, kms = np.array(lat[3:]) * 1e3, np.array(kms[3:])
n_pts = int(pl.engine.points_per_query(np.array([[5.0, 5.0, 0.0, 0.0, 0.0, 0.0]]), np.array([6])).sum())
out["config2"] = {"plan_ms_p50": float(np.median(lat)), "plan_ms_p95": float(np.percentile(lat, 95)),
                  "kernel_ms_p50": float(np.median(kms)), "candidates": 1261, "dense_evals": n_pts * 50,
                  "winner_index": None if path is None else int(pl.last_result.best_idx[0])}

# ---- config 3 ---------------------------------------------------------------------------------
rng = np.random.default_rng(33)
knobs = dict(k, d_road_w=0.1, max_road_width=3.2, min_t=1.9, max_t=5.0, d_t_s=0.2)
wp = (np.linspace(0.0, 80.0, 9).tolist(), [0.0] * 9)
base = scenarios.pedestrian_field(rng, 200, x_range=(5.0, 65.0), vel_clip=2.5)
dist = scenarios.sample_distribution(rng, base, 20)
bp = BatchFrenetPlanner(CubicSpline2D(*wp), **knobs)
fs = np.array([[5.0, 5.0, 0.0, 0.0, 0.0, 0.0]])
res3 = {}
for kern in ("pairs", "items"):
    os.environ["FOT_SWEEP"] = kern
    bp.engine.reload_options()
    ms = []
    for _ in range(6):
        r = bp.plan_batch(fs, 6.2, distribution=dist[None])
        ms.append(r.kernel_ms)
    res3[kern + "_kernel_ms"] = float(np.median(ms[1:]))
os.environ.pop("FOT_SWEEP")
bp.engine.reload_options()
from integrated_path_planning_b200.engine import speed_grid
pts = int(bp.engine.points_per_query(fs, np.array([len(speed_grid(6.2, knobs["d_t_s"]))])).sum())
res3.update({"candidates": int(r.n_cand[0]), "dense_evals": pts * 4000, "stats": r.stats[0].tolist()})
res3["dense_evals_per_s_items"] = res3["dense_evals"] / (res3["items_kernel_ms"] * 1e-3)
out["config3"] = res3

# ---- config 5 ---------------------------------------------------------------------------------
plans = [(6.0, None, None),
         (3.6, {"max_accel": k["max_accel"] * 1.5, "max_speed": k["max_speed"] * 0.6}, None),
         (0.0, {"max_accel": k["max_accel"] * 3.0, "max_lat_accel": k["max_lat_accel"] * 2.0}, 5.0)]
pl = FrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **k)
rng = np.random.default_rng(17)
ego = np.array([3.0, 0.1, 0.0, 5.0, 0.0])
step_ms, found = [], 0
for step in range(500):
    dyn = scenarios.pedestrian_field(rng, 10, x_range=(ego[0] + 3, ego[0] + 30), y_range=(-6, 6))
    t0 = time.perf_counter()
    for target, ovr, msd in plans:
        path = pl.plan(runners._Ego(*ego), static, dyn, target, ovr, None, msd)
        found += path is not None
    step_ms.append((time.perf_counter() - t0) * 1e3)
    ego = ego + np.array([0.09, rng.normal(0, 0.02), rng.normal(0, 0.005), rng.normal(0, 0.1), 0.0])
    ego[0] = 3.0 + (ego[0] - 3.0) % 20.0
step_ms = np.array(step_ms[5:])
out["config5"] = {"steps": 500, "plans_per_step": 3, "step_ms_p50": float(np.median(step_ms)),
                  "step_ms_p95": float(np.percentile(step_ms, 95)), "paths_found": int(found)}
print(json.dumps(out))
