#!/usr/bin/env python
"""Multi-route batches: what a per-query route costs on a resident config-4 launch.

    python tools/bench_routes.py --queries 4096 --steps 100 --warmup 5 --out profiles/r3/bench_routes.json

The config-4 queries of bench.py (4096 resident queries, 50 pedestrians each) go through `DeviceBatch` in variants that
alternate in one process, every step timed with CUDA events on one stream:
  unrouted      the launch bench.py times (no route binding);
  routed_R      the same queries spread over R distinct routes (R in 1, 8, 64; query q on route q % R), one launch;
  separate_R    what a caller without routes does: R planners, one per path, each launching its own N/R queries, in
                sequence (the whole sequence is one step).
  closed_loop   a BatchedClosedLoop lock-step of 192 simulations over three routes (scenario_01's road, scenario_03's
                right turn, an S-curve; 64 each), against three single-route loops of 64 simulations stepped one after
                the other: host wall-clock per lock-step (every simulation advanced once), 60 steps after warm-up, second of
                two rounds.
Routes are the straight 60 m line of config 4 and gently curved variants of it, 20 knots each (every one <= 48 knots,
so fot_sweep_pairs runs).  `stages_ms` is the median fot_launch_stage_ms breakdown (prepass, sweep, winner) of a
variant's launches.  After the timed steps every routed variant's winners must equal, bit for bit, those of the
separate per-route launches.  Prints one JSON line with the card's name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def route_waypoints(r: int):
    """Route 0: config 4's straight line; route r > 0: a gentle S-bend of that line, 20 knots."""
    from tests import scenarios
    if r == 0:
        return scenarios.STRAIGHT_60
    x = np.linspace(0.0, 60.0 + 0.25 * (r % 7), 20)
    amp = 0.05 + 0.02 * r
    return x.tolist(), (amp * np.sin(2 * np.pi * x / (40.0 + r % 13))).tolist()


def closed_loop(n_per_route: int = 64, n_steps: int = 60):
    """(ms per lock-step of one routed loop, of three single-route loops in sequence, histories equal)."""
    import time
    from tests import runners, scenarios
    from integrated_path_planning_b200 import CubicSpline2D
    from integrated_path_planning_b200.rollout import BatchedClosedLoop
    z, z3 = runners.load_golden("rollout_s01.npz"), runners.load_golden("rollout_s03.npz")
    knobs = {k[5:]: float(z[k]) for k in z.files if k.startswith("knob/")}
    paths = [(z["v0/wx"], z["v0/wy"]), (z3["v0/wx"], z3["v0/wy"]), scenarios.s_curve_waypoints(length=80.0, amp=3.0, n=20)]
    starts = []
    for wx, wy in paths:
        sp = CubicSpline2D(list(wx), list(wy))
        x, y = sp.calc_position(0.0)
        starts.append([float(x), float(y), float(sp.calc_yaw(0.0)), 5.0, 0.0])
    route = np.arange(3 * n_per_route) % 3
    tracks = np.stack([z[f"v{i % 4}/traj"] for i in range(len(route))])
    ego0 = np.array([starts[r] for r in route])

    def drive(sim):
        sim.warmup()
        sim.step()                                          # first step: handle, buffers
        t0 = time.perf_counter()
        out = sim.run(n_steps)
        return out, (time.perf_counter() - t0) * 1e3 / n_steps
    # two rounds, routed then single-route; the second (warm) round is reported: the first pays the process's module
    # loads and allocator growth
    for _ in range(2):
        routed, ms_routed = drive(BatchedClosedLoop(paths[0][0], paths[0][1], knobs, tracks, ego0, routes=paths[1:],
                                                    route=route))
        ms_single, same = 0.0, True
        for r, (wx, wy) in enumerate(paths):
            rows = np.nonzero(route == r)[0]
            out, ms = drive(BatchedClosedLoop(wx, wy, knobs, tracks[rows], ego0[rows]))
            ms_single += ms
            same &= all(np.array_equal(routed[k][rows], out[k], equal_nan=k == "ego")          # NaN: steps after the end
                        for k in ("ego", "fsm", "found", "calls", "steps"))
    return {"simulations": int(len(route)), "routes": 3, "steps": n_steps, "ms_per_lockstep_routed": ms_routed,
            "ms_per_lockstep_three_single_route_loops": ms_single, "histories_equal": bool(same)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=100, help="timed steps per variant, in rounds of --block")
    ap.add_argument("--block", type=int, default=20, help="consecutive steps of one variant before the next one runs")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--routes", default="1,8,64")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    import bench
    from tests import scenarios
    from integrated_path_planning_b200 import CubicSpline2D, _lib
    from integrated_path_planning_b200.batch import BatchFrenetPlanner, DeviceBatch
    if not torch.cuda.is_available():
        raise SystemExit("bench_routes.py needs a CUDA device")
    n_q = args.queries
    counts = [int(v) for v in args.routes.split(",")]
    _, frenet, dyn = bench.make_queries(0, n_q)
    dyn_d = torch.from_numpy(dyn).cuda()
    new_planner = lambda r: BatchFrenetPlanner(CubicSpline2D(*route_waypoints(r)), **scenarios.S1_KNOBS)
    base = new_planner(0)
    variants = {"unrouted": [(base.engine, DeviceBatch(base, frenet, bench.TARGET_SPEED, dyn_d, _lib.FOT_DYN_SINGLE))]}
    rows_of = {}
    for R in counts:
        pl = new_planner(0)
        for r in range(1, R):
            pl.add_route(CubicSpline2D(*route_waypoints(r)))
        route = np.arange(n_q) % R
        variants[f"routed_{R}"] = [(pl.engine, DeviceBatch(pl, frenet, bench.TARGET_SPEED, dyn_d, _lib.FOT_DYN_SINGLE,
                                                            route=route))]
        sep = []
        for r in range(R):
            rows = np.nonzero(route == r)[0]
            rows_of[(R, r)] = rows
            p = new_planner(r)
            sep.append((p.engine, DeviceBatch(p, frenet[rows], bench.TARGET_SPEED, dyn_d[torch.from_numpy(rows).cuda()],
                                              _lib.FOT_DYN_SINGLE)))
        variants[f"separate_{R}"] = sep
    stream = torch.cuda.Stream()
    raw = stream.cuda_stream

    def step(launches, ev):
        ev[0].record(stream)
        for eng, db in launches:
            with eng.routes_bound(db._route_ptr()):
                eng.run_device(db.batch, db.result, raw)
        ev[1].record(stream)

    new_ev = lambda: [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    times = {name: [] for name in variants}
    stages = {name: [] for name in variants}
    with torch.cuda.stream(stream):
        for name, launches in variants.items():
            for _ in range(args.warmup):
                step(launches, new_ev())
        stream.synchronize()
        for _ in range(max(1, -(-args.steps // args.block))):
            for name, launches in variants.items():
                evs = [new_ev() for _ in range(args.block)]
                for ev in evs:
                    step(launches, ev)
                stream.synchronize()
                times[name] += [ev[0].elapsed_time(ev[1]) for ev in evs]
                if len(launches) == 1:
                    eng = launches[0][0]
                    stages[name] += [eng.launch_stage_ms(b) for b in range(min(args.block, 256))]
    out = {}
    for name, launches in variants.items():
        t = np.array(times[name])
        row = {"launches_per_step": len(launches), "steps": len(t), "ms_per_step": float(np.median(t)),
               "ms_per_step_p10_p90": [float(np.percentile(t, 10)), float(np.percentile(t, 90))]}
        if stages[name]:
            row["stages_ms"] = dict(zip(("prepass", "sweep", "winner"), np.median(np.array(stages[name]), axis=0).tolist()))
            eng = launches[0][0]
            row["sweep_kind"], row["pair_features"] = int(eng.lib.fot_last_sweep_kind(eng._h)), \
                int(eng.lib.fot_last_pair_features(eng._h))
        out[name] = row
    # routed winners == the separate per-route launches, bit for bit
    same = {}
    for R in counts:
        o = {k: v.cpu().numpy() for k, v in variants[f"routed_{R}"][0][1].out.items()}
        ok = True
        for r, (_, db) in enumerate(variants[f"separate_{R}"]):
            rows, p = rows_of[(R, r)], {k: v.cpu().numpy() for k, v in db.out.items()}
            ok &= all(np.array_equal(o[k][rows], p[k]) for k in ("best_idx", "stats", "winner_len"))
            ok &= np.array_equal(o["best_cost"][rows].view(np.uint64), p["best_cost"].view(np.uint64))
            live = np.arange(o["winner"].shape[-1])[None, None, :] < p["winner_len"].reshape(-1, 1, 1)
            ok &= np.array_equal(np.where(live, o["winner"][rows], 0.0).view(np.uint64),
                                 np.where(live, p["winner"], 0.0).view(np.uint64))
        same[R] = bool(ok)
        out[f"routed_{R}"]["winners_equal_separate_launches"] = bool(ok)
    loop = closed_loop()
    result = {"tool": "bench_routes", "card": card(), "queries": n_q, "route_knots": 20, "variants": out, "closed_loop": loop}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    assert all(same.values()) and loop["histories_equal"], (same, loop)


if __name__ == "__main__":
    main()
