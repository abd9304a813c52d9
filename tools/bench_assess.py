#!/usr/bin/env python
"""Trajectory assessment: what fot_assess_trajectories costs behind a resident config-4 launch.

    python tools/bench_assess.py --queries 4096 --steps 100 --warmup 5 --out profiles/r3/bench_assess.json

The config-4 queries of bench.py (4096 resident queries, 50 pedestrians, 51 obstacle steps) go through `DeviceBatch`
in five variants that alternate in one process, in blocks of --block steps:
  plain            the launch bench.py times
  winners_own      + assessment of the winners against their own tensor                 (case a)
  top8             top_k = 8 ranked alternatives with series
  top8_assessed    + assessment of the 8 alternatives against their own tensor          (case b)
  winners_dist20   + assessment of the winners against a 20-sample distribution of the same pedestrians (case c)
Every step is timed with CUDA events on one stream: `launch_ms` covers fot_plan_batch_device (and fot_rank_candidates),
`assess_ms` the fot_assess_trajectories call alone.  `extra_ms_per_step` is a variant's median step time less that of
the variant it extends.  The bytes the kernel must read are computed from shapes and the slot lengths of the run:
the obstacle tensor once for every query with a live slot (the kernel blanks a query without one and never reads its
tensor), the rows t, x, y, yaw of every live sample, the lengths and thresholds; the outputs it writes are counted
apart.  `hbm_share` is those bytes at 7.7 TB/s (the B200's HBM3e bandwidth) over the kernel time.  After the
timed steps the winner blocks of every variant must equal the plain launch's, and every assessed winner must be
collision-free under the handle's own pair against its own tensor.  Prints one JSON line with the card's name and
power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def read_bytes(lens, S, P, T, n_r):
    """Bytes fot_assess must read and write for slot lengths lens [n_q, m]: the obstacle tensor once for every query
    with a live slot (a query whose slots are all empty is blanked without reading it), the four series rows t, x, y,
    yaw of every live sample, every slot's length and the thresholds; and the outputs of every slot."""
    n_q, m = lens.shape
    live_q = int((lens > 0).any(axis=1).sum())
    reads = live_q * S * P * T * 16 + int(lens.sum()) * 4 * 8 + n_q * m * 4 + n_r * 16
    writes = n_q * m * (8 + 16 + 8 + 12 + 3 * 4 * n_r)
    return int(reads), int(writes), live_q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=100, help="timed steps per variant, in rounds of --block")
    ap.add_argument("--block", type=int, default=20, help="consecutive steps of one variant before the next one runs")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--samples", type=int, default=20, help="samples of the distribution of case c")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    import bench
    from tests import scenarios
    from integrated_path_planning_b200 import _lib
    from integrated_path_planning_b200.batch import BatchFrenetPlanner, DeviceBatch
    from integrated_path_planning_b200 import CubicSpline2D
    if not torch.cuda.is_available():
        raise SystemExit("bench_assess.py needs a CUDA device")
    planner = BatchFrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    _, frenet, dyn = bench.make_queries(0, args.queries)
    dev = torch.device("cuda", planner.engine.device)
    dyn_d = torch.from_numpy(dyn).to(dev)
    # case c: the same pedestrians as S samples, each a random walk away from the CV track (zero at step 0), on the device
    gen = torch.Generator(device=dev).manual_seed(7)
    walk = torch.randn((args.queries, args.samples) + tuple(dyn.shape[2:]), generator=gen, device=dev,
                       dtype=torch.float64) * 0.05
    walk[:, :, :, 0] = 0.0
    dist_d = (dyn_d[:, :1] + torch.cumsum(walk, dim=3)).contiguous()
    del walk
    S1 = _lib.FOT_DYN_SINGLE
    variants = {
        "plain": (None, dict()),
        "winners_own": ("plain", dict(assess=True)),
        "top8": (None, dict(top_k=8)),
        "top8_assessed": ("top8", dict(top_k=8, assess=True)),
        "winners_dist20": ("plain", dict(assess=True, assess_obstacles=dist_d)),
    }
    batches = {name: DeviceBatch(planner, frenet, bench.TARGET_SPEED, dyn_d, S1, **kw) for name, (_, kw) in variants.items()}
    stream = torch.cuda.Stream(dev)
    raw = stream.cuda_stream
    eng = planner.engine

    def step(db, ev):
        ev[0].record(stream)
        eng.run_device(db.batch, db.result, raw)
        if db.top_k > 0:
            r = db.result
            eng.rank_device(db.batch, r.cand_cat, r.cand_cost, r.cand_stride, db.ranked, raw)
        ev[1].record(stream)
        if db.assess:
            eng.assess_device(db.assess_field, db.assessed, raw)
        ev[2].record(stream)

    new_ev = lambda: [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    with torch.cuda.stream(stream):
        for name in variants:
            for _ in range(args.warmup):
                step(batches[name], new_ev())
        stream.synchronize()
        times = {name: [] for name in variants}
        for _ in range(max(1, -(-args.steps // args.block))):
            for name in variants:
                evs = [new_ev() for _ in range(args.block)]
                for ev in evs:
                    step(batches[name], ev)
                stream.synchronize()
                times[name] += [(ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[0].elapsed_time(ev[2]))
                                for ev in evs]
    host = {name: {k: v.cpu().numpy() for k, v in db.out.items()} for name, db in batches.items()}
    ref = host["plain"]
    n_q, T, P = args.queries, dyn.shape[3], dyn.shape[2]
    out = {}
    for name, (base, kw) in variants.items():
        t = np.array(times[name])
        db = batches[name]
        row = {"steps": len(t), "ms_per_step": float(np.median(t[:, 2])), "launch_ms": float(np.median(t[:, 0])),
               "ms_per_step_p10_p90": [float(np.percentile(t[:, 2], 10)), float(np.percentile(t[:, 2], 90))]}
        o = host[name]
        same = all(np.array_equal(o[k], ref[k]) for k in ("best_idx", "stats", "winner_len"))
        same &= np.array_equal(o["best_cost"].view(np.uint64), ref["best_cost"].view(np.uint64))
        row["winners_unchanged"] = bool(same)
        if db.assess:
            a = db.assessed
            S = args.samples if "assess_obstacles" in kw else 1
            lens = o["rank_len" if a.m > 1 else "winner_len"].reshape(n_q, -1)
            reads, writes, live_q = read_bytes(lens, S, P, T, a.n_r)
            kernel = float(np.median(t[:, 1]))
            row.update(assess_ms=kernel, assess_ms_p10_p90=[float(np.percentile(t[:, 1], 10)),
                                                             float(np.percentile(t[:, 1], 90))],
                       m=int(a.m), S=S, queries_read=live_q, bytes_read=reads, bytes_written=writes,
                       hbm_share=(reads + writes) / HBM_BYTES_PER_S / (kernel * 1e-3),
                       extra_ms_per_step=row["ms_per_step"] - float(np.median(np.array(times[base])[:, 2])))
            live = lens > 0
            row["assessed_trajectories"] = int(live.sum())
            if S == 1:      # against its own tensor every returned trajectory is collision-free under the own pair
                row["all_collision_free"] = bool(np.all(o["a_dyn_hits"][live][:, 0] == 0) and
                                                 np.all(o["a_static_hit"][live][:, 0] == 0))
            else:
                hits = o["a_dyn_hits"][live][:, 0]
                row["hit_fraction_mean"] = float(np.mean(hits / S)) if hits.size else 0.0
                row["trajectories_hitting_some_sample"] = int((hits > 0).sum())
        out[name] = row
    result = {"tool": "bench_assess", "card": card(), "queries": n_q, "pedestrians": int(P), "obstacle_steps": int(T),
              "n_t_max": int(eng.n_t_max), "hbm_bytes_per_s": HBM_BYTES_PER_S, "variants": out}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    assert all(v["winners_unchanged"] for v in out.values()), "an assessed launch changed the winners"
    assert all(v.get("all_collision_free", True) for v in out.values()), "a returned trajectory collides"


if __name__ == "__main__":
    main()
