#!/usr/bin/env python
"""Ranked alternatives: what ranking costs on top of a resident config-4 launch.

    python tools/bench_ranked.py --queries 4096 --steps 100 --warmup 5 --out profiles/r3/bench_ranked.json

The config-4 queries of bench.py (4096 resident queries, 50 pedestrians each) go through `DeviceBatch` in seven
variants that alternate in one process: the plain launch (what bench.py times), and top_k in {1, 8, 32} with the
series on and off.  Every step is timed with CUDA events on one stream: `sweep` is the fot_plan_batch_device launch
(prepass, sweep kernel, winner kernel; the ranked variants run the sweep instantiation that writes the per-candidate
table), `rank` the fot_rank_candidates call (fot_rank, plus fot_rank_series when the series are on).  `series_ms` is
the series variant's rank time less the same top_k without series.  After the timed steps every ranked variant's
rank 0 must be the winner of its own launch (index, cost bits, length, series bits) and its winner block must equal
the plain launch's.  Prints one JSON line with the card's name and power limit, read in the same run.
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


def check(db, plain):
    """Rank 0 is the winner of the same launch, and the winner block is the plain launch's."""
    o, p = {k: v.cpu().numpy() for k, v in db.out.items()}, {k: v.cpu().numpy() for k, v in plain.out.items()}
    ok = all(np.array_equal(o[k], p[k]) for k in ("best_idx", "stats", "winner_len"))
    ok &= np.array_equal(o["best_cost"].view(np.uint64), p["best_cost"].view(np.uint64))
    ok &= np.array_equal(o["rank_idx"][:, 0], o["best_idx"])
    ok &= np.array_equal(o["rank_cost"][:, 0].view(np.uint64), o["best_cost"].view(np.uint64))
    rows = np.nonzero(o["best_idx"] >= 0)[0]
    n_t = o["winner"].shape[-1]
    live = np.arange(n_t)[None, None, :] < o["winner_len"][rows].reshape(-1, 1, 1)
    ok &= np.array_equal(np.where(live, o["winner"][rows], 0.0).view(np.uint64),
                         np.where(live, p["winner"][rows], 0.0).view(np.uint64))
    if "rank_series" in o:
        ok &= np.array_equal(o["rank_len"][:, 0], o["winner_len"])
        ok &= np.array_equal(np.where(live, o["rank_series"][rows, 0], 0.0).view(np.uint64),
                             np.where(live, o["winner"][rows], 0.0).view(np.uint64))
    return bool(ok), int(len(rows))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=100, help="timed steps per variant (>= 50), in rounds of --block")
    ap.add_argument("--block", type=int, default=20, help="consecutive steps of one variant before the next one runs")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    import bench
    from tests import scenarios
    from integrated_path_planning_b200 import _lib
    from integrated_path_planning_b200.batch import BatchFrenetPlanner, DeviceBatch
    from integrated_path_planning_b200 import CubicSpline2D
    if not torch.cuda.is_available():
        raise SystemExit("bench_ranked.py needs a CUDA device")
    planner = BatchFrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    _, frenet, dyn = bench.make_queries(0, args.queries)
    dyn_d = torch.from_numpy(dyn).cuda()
    variants = [("plain", 0, False)] + [(f"top{k}_{'series' if s else 'noseries'}", k, s)
                                        for k in (1, 8, 32) for s in (False, True)]
    batches = {name: DeviceBatch(planner, frenet, bench.TARGET_SPEED, dyn_d, _lib.FOT_DYN_SINGLE, top_k=k, rank_series=s)
               for name, k, s in variants}
    stream = torch.cuda.Stream()
    raw = stream.cuda_stream
    eng = planner.engine

    def step(db, ev):
        ev[0].record(stream)
        eng.run_device(db.batch, db.result, raw)
        ev[1].record(stream)
        if db.top_k > 0:
            r = db.result
            eng.rank_device(db.batch, r.cand_cat, r.cand_cost, r.cand_stride, db.ranked, raw)
        ev[2].record(stream)

    new_ev = lambda: [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    with torch.cuda.stream(stream):
        for name, _, _ in variants:
            for _ in range(args.warmup):
                step(batches[name], new_ev())
        stream.synchronize()
        times = {name: [] for name, _, _ in variants}
        rounds = max(1, -(-args.steps // args.block))
        for _ in range(rounds):
            for name, _, _ in variants:
                evs = [new_ev() for _ in range(args.block)]
                for ev in evs:
                    step(batches[name], ev)
                stream.synchronize()
                times[name] += [(ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[0].elapsed_time(ev[2]))
                                for ev in evs]
    plain = batches["plain"]
    out = {}
    for name, k, s in variants:
        t = np.array(times[name])
        row = {"top_k": k, "series": s, "steps": len(t), "ms_per_step": float(np.median(t[:, 2])),
               "sweep_ms": float(np.median(t[:, 0])), "rank_ms": float(np.median(t[:, 1])),
               "ms_per_step_p10_p90": [float(np.percentile(t[:, 2], 10)), float(np.percentile(t[:, 2], 90))]}
        if k > 0:
            row["rank0_is_winner_and_winners_unchanged"], row["queries_with_winner"] = check(batches[name], plain)
        out[name] = row
    for k in (1, 8, 32):
        on, off = out[f"top{k}_series"], out[f"top{k}_noseries"]
        on["series_ms"] = on["rank_ms"] - off["rank_ms"]
    n_q = args.queries
    stride = int(plain.engine.lib.fot_candidate_count(eng._h, int(plain.batch.n_v_max), 1))
    result = {"tool": "bench_ranked", "card": card(), "queries": n_q, "candidates_per_query": stride,
              "table_bytes": n_q * stride * 9,
              "series_bytes_written_at_k": {k: n_q * k * _lib.FOT_N_SERIES * eng.n_t_max * 8 for k in (1, 8, 32)},
              "variants": out}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    assert all(v.get("rank0_is_winner_and_winners_unchanged", True) for v in out.values()), "rank 0 != winner"


if __name__ == "__main__":
    main()
