#!/usr/bin/env python
"""Planning from ego states: the nearest-point search on the device against the host converter.

    python tools/bench_from_ego.py --queries 4096 --reps 7 --sims 256 --steps 30

Everything runs in one process and each pair of variants alternates rep by rep:
  cold      the config-4 egos of bench.py (`ego_and_field`), each with a fresh converter (no cache: global search):
            ego -> Frenet time with the host converter and with the engine-backed one, the share of rows the device
            left to the host, and `plan_batch_from_ego` end to end against host conversion + `plan_batch`;
  warm      the same egos one step (v * dt) along the path, with the caches the cold call left (cached window);
  rollout   a 256-simulation BatchedClosedLoop lock-step (tools/bench_rollout.py's campaign), host converters against
            engine-backed ones.
Every pair of outputs is compared bit for bit at the timed size.  Prints one JSON line with the card's name and power
limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return time.perf_counter() - t0, out


def same(a, b):
    return bool(np.array_equal(a, b, equal_nan=True))


def conversion(args, planner, spline, ego, kappa):
    from integrated_path_planning_b200.frenet_host import BatchCoordinateConverter, ego_to_frenet_many
    n = len(ego)
    idx = np.arange(n)
    t = {"host": [], "device": []}
    out = {}
    for _ in range(args.reps):
        for kind in ("host", "device"):
            conv = BatchCoordinateConverter(spline, n, engine=planner.engine if kind == "device" else None)
            dt, res = timed(lambda: ego_to_frenet_many(conv, idx, ego, kappa))
            t[kind].append(dt)
            out[kind] = (res, conv)
    (fs_h, ok_h), conv_h = out["host"]
    (fs_d, ok_d), conv_dev = out["device"]
    cold = {"ms_host": 1e3 * float(np.median(t["host"])), "ms_device": 1e3 * float(np.median(t["device"])),
            "status1_share": conv_dev.host_rows / max(1, conv_dev.host_rows + conv_dev.device_rows),
            "equal": same(fs_h, fs_d) and same(ok_h, ok_d) and same(conv_h.prev_s, conv_dev.prev_s)}

    # one step along the path from the cached positions
    step = ego.copy()
    step[:, 0] += ego[:, 3] * np.cos(ego[:, 2]) * 0.1
    step[:, 1] += ego[:, 3] * np.sin(ego[:, 2]) * 0.1
    warm_prev = conv_h.prev_s.copy()
    t = {"host": [], "device": []}
    for _ in range(args.reps):
        for kind in ("host", "device"):
            conv = BatchCoordinateConverter(spline, n, engine=planner.engine if kind == "device" else None)
            conv.prev_s[:] = warm_prev
            dt, res = timed(lambda: ego_to_frenet_many(conv, idx, step, kappa))
            t[kind].append(dt)
            out[kind] = (res, conv)
    (fs_h, ok_h), conv_h = out["host"]
    (fs_d, ok_d), conv_d = out["device"]
    warm = {"ms_host": 1e3 * float(np.median(t["host"])), "ms_device": 1e3 * float(np.median(t["device"])),
            "status1_share": conv_d.host_rows / max(1, conv_d.host_rows + conv_d.device_rows),
            "equal": same(fs_h, fs_d) and same(ok_h, ok_d) and same(conv_h.prev_s, conv_d.prev_s)}
    return cold, warm


def end_to_end(args, planner, spline, ego, kappa, dyn, target):
    from integrated_path_planning_b200.frenet_host import BatchCoordinateConverter, ego_to_frenet_many
    n = len(ego)
    keys = ("best_idx", "best_cost", "stats", "winner_len", "winner")

    def host():
        fs, ok = ego_to_frenet_many(BatchCoordinateConverter(spline, n), np.arange(n), ego, kappa)
        res = planner.plan_batch(fs, target, dynamic_obstacles=dyn)
        return {k: getattr(res, k).copy() for k in keys}

    def device():
        res, ok = planner.plan_batch_from_ego(ego, target, last_kappa=kappa, dynamic_obstacles=dyn)
        return {k: getattr(res, k).copy() for k in keys}

    host(), device()                                   # warm-up: pinned buffers, speed grid, kernels
    t = {"host": [], "device": []}
    out = {}
    for _ in range(args.reps):
        for kind, fn in (("host", host), ("device", device)):
            dt, out[kind] = timed(fn)
            t[kind].append(dt)
    equal = all(same(out["host"][k].view(np.int64) if out["host"][k].dtype == np.float64 else out["host"][k],
                     out["device"][k].view(np.int64) if out["device"][k].dtype == np.float64 else out["device"][k])
                for k in keys[:4])
    ok_rows = out["host"]["best_idx"] >= 0
    equal &= all(same(out["host"]["winner"][q, :, :out["host"]["winner_len"][q]],
                      out["device"]["winner"][q, :, :out["device"]["winner_len"][q]]) for q in np.nonzero(ok_rows)[0])
    return {"ms_host_conversion_plus_plan_batch": 1e3 * float(np.median(t["host"])),
            "ms_plan_batch_from_ego": 1e3 * float(np.median(t["device"])), "equal": bool(equal)}


def rollout(args):
    from integrated_path_planning_b200.frenet_host import BatchCoordinateConverter
    from integrated_path_planning_b200.rollout import BatchedClosedLoop
    z = np.load(os.path.join(ROOT, "tests", "golden", "rollout_s01.npz"))
    knobs = {k[5:]: float(z[k]) for k in z.files if k.startswith("knob/")}
    rng = np.random.default_rng(7)
    n_var = int(z["n_variants"])
    tracks, ego0 = [], []
    for i in range(args.sims):
        v = i % n_var
        t = z[f"v{v}/traj"]
        tracks.append(t + rng.normal(0.0, 0.3, (1, t.shape[1], 2)))
        e = z[f"v{v}/ego0"].copy()
        e[3] = max(0.5, e[3] + rng.normal(0.0, 0.3))
        ego0.append(e)
    sims = {}
    for kind in ("host", "device"):
        sim = BatchedClosedLoop(z["v0/wx"], z["v0/wy"], knobs, np.stack(tracks), np.stack(ego0))
        if kind == "host":
            sim.plan_conv = BatchCoordinateConverter(sim.spline, sim.n)
            sim.goal_conv = BatchCoordinateConverter(sim.spline, sim.n)
        sim.warmup()
        for _ in range(3):
            sim.step()
        sims[kind] = sim
    t = {"host": [], "device": []}
    equal = True
    for _ in range(args.steps):
        for kind in ("host", "device"):
            dt, _ = timed(sims[kind].step)
            t[kind].append(dt)
        equal &= same(sims["host"].ego, sims["device"].ego) and same(sims["host"].active, sims["device"].active)
    d = sims["device"]
    rows = d.plan_conv.host_rows + d.plan_conv.device_rows + d.goal_conv.host_rows + d.goal_conv.device_rows
    return {"sims": args.sims, "steps": args.steps, "ms_per_lockstep_host": 1e3 * float(np.median(t["host"])),
            "ms_per_lockstep_device": 1e3 * float(np.median(t["device"])),
            "status1_share": (d.plan_conv.host_rows + d.goal_conv.host_rows) / max(1, rows),
            "still_active": int(d.active.sum()), "equal": bool(equal)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--sims", type=int, default=256)
    ap.add_argument("--steps", type=int, default=30)
    args = ap.parse_args()
    import bench
    from tests import scenarios
    from integrated_path_planning_b200 import CubicSpline2D
    from integrated_path_planning_b200.batch import BatchFrenetPlanner
    spline = CubicSpline2D(*scenarios.STRAIGHT_60)
    planner = BatchFrenetPlanner(spline, **scenarios.S1_KNOBS)
    n = args.queries
    ego = np.empty((n, 5))
    dyn = np.empty((n, bench.N_PEDS, bench.T_OBS, 2))
    for i in range(n):
        e, d = bench.ego_and_field(i)
        ego[i], dyn[i] = e, d
    kappa = np.zeros(n)
    planner.engine.nearest_s(ego[:32, 0], ego[:32, 1], np.full(32, np.nan))   # module load, staging buffers
    cold, warm = conversion(args, planner, spline, ego, kappa)
    e2e = end_to_end(args, planner, spline, ego, kappa, dyn, bench.TARGET_SPEED)
    roll = rollout(args)
    print(json.dumps({"tool": "bench_from_ego", "card": card(), "queries": n, "reps": args.reps,
                      "conversion_cold": cold, "conversion_warm": warm, "end_to_end": e2e, "rollout": roll}))


if __name__ == "__main__":
    main()
