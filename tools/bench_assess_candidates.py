#!/usr/bin/env python
"""Candidate assessment: what fot_assess_candidates costs behind a resident config-4 launch.

    python tools/bench_assess_candidates.py --queries 4096 --steps 40 --warmup 3 --out profiles/r3/bench_assess_candidates.json

The config-4 queries of bench.py (4096 resident queries, 1261 candidates each, 50 pedestrians, 51 obstacle steps) go
through `DeviceBatch` in three variants that alternate in one process, in blocks of --block steps:
  plain         the launch bench.py times
  cand_own      + every candidate assessed against its query's own tensor (S = 1)
  cand_dist20   + every candidate assessed against a 20-sample distribution of the same pedestrians
(The categories come from a separate, untimed launch that also writes the per-candidate table.)
Every step is timed with CUDA events on one stream: `launch_ms` covers fot_plan_batch_device, `assess_ms` the
fot_assess_candidates call alone (its NaN-bit pass and the kernel).  `extra_ms_per_step` is a variant's median step time
less the plain launch's.  `dense_tests` are the distance tests the kernel must do: the kept samples of every candidate
(Sum keep) times the circles times (S*P + M); `tests_per_s` is that over the kernel time, and `fma_share` that rate over
the FP64 FMA rate fot_probe_fma_tflops measures in the same run (FMAs/s = TFLOP/s / 2).  `bytes_moved` counts the
obstacle tensor twice (the NaN-bit pass and the kernel's reads, once per query), the query arrays and every output;
`hbm_share` is that at 7.7 TB/s over the kernel time.  After the timed steps the winner blocks of every variant must
equal the plain launch's, and under the handle's own pair the category of every candidate must agree with its
assessment against its own tensor.  Prints one JSON line with the card's name and power limit, read in the same run.
"""
import argparse
import ctypes
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=40, help="timed steps per variant, in rounds of --block")
    ap.add_argument("--block", type=int, default=10, help="consecutive steps of one variant before the next one runs")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--samples", type=int, default=20, help="samples of the distribution of cand_dist20")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    import bench
    from tests import scenarios
    from integrated_path_planning_b200 import _lib
    from integrated_path_planning_b200.batch import BatchFrenetPlanner, DeviceBatch
    from integrated_path_planning_b200 import CubicSpline2D
    if not torch.cuda.is_available():
        raise SystemExit("bench_assess_candidates.py needs a CUDA device")
    planner = BatchFrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    _, frenet, dyn = bench.make_queries(0, args.queries)
    eng = planner.engine
    dev = torch.device("cuda", eng.device)
    dyn_d = torch.from_numpy(dyn).to(dev)
    gen = torch.Generator(device=dev).manual_seed(7)
    walk = torch.randn((args.queries, args.samples) + tuple(dyn.shape[2:]), generator=gen, device=dev,
                       dtype=torch.float64) * 0.05
    walk[:, :, :, 0] = 0.0
    dist_d = (dyn_d[:, :1] + torch.cumsum(walk, dim=3)).contiguous()
    del walk
    variants = {
        "plain": dict(),
        "cand_own": dict(assess_candidates=True),
        "cand_dist20": dict(assess_candidates=True, assess_obstacles=dist_d),
    }
    batches = {name: DeviceBatch(planner, frenet, bench.TARGET_SPEED, dyn_d, _lib.FOT_DYN_SINGLE, **kw)
               for name, kw in variants.items()}
    stream = torch.cuda.Stream(dev)
    raw = stream.cuda_stream

    def step(db, ev):
        ev[0].record(stream)
        eng.run_device(db.batch, db.result, raw)
        ev[1].record(stream)
        if db.assess_candidates:
            eng.assess_candidates_device(db.batch, db.assess_field, db.stride, db.cand_assessed,
                                         db.out["ca_keep"].data_ptr(), raw)
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
    fma = ctypes.c_double()
    _lib.check(eng.lib.fot_probe_fma_tflops(eng.device, 0, ctypes.byref(fma)), "fot_probe_fma_tflops")
    fma_per_s = fma.value * 1e12 / 2
    host = {name: {k: v.cpu().numpy() for k, v in db.out.items()} for name, db in batches.items()}
    ref = host["plain"]
    n_q, P, T = args.queries, dyn.shape[2], dyn.shape[3]
    nc = max(1, eng.n_circles)
    plain_ms = float(np.median(np.array(times["plain"])[:, 2]))
    out = {}
    for name, kw in variants.items():
        t = np.array(times[name])
        db = batches[name]
        row = {"steps": len(t), "ms_per_step": float(np.median(t[:, 2])), "launch_ms": float(np.median(t[:, 0])),
               "ms_per_step_p10_p90": [float(np.percentile(t[:, 2], 10)), float(np.percentile(t[:, 2], 90))]}
        o = host[name]
        same = all(np.array_equal(o[k], ref[k]) for k in ("best_idx", "stats", "winner_len"))
        same &= np.array_equal(o["best_cost"].view(np.uint64), ref["best_cost"].view(np.uint64))
        row["winners_unchanged"] = bool(same)
        if db.assess_candidates:
            S = args.samples if "assess_obstacles" in kw else 1
            keep = o["ca_keep"].astype(np.int64)
            kernel = float(np.median(t[:, 1]))
            dense = int(keep.sum()) * nc * (S * P + db.batch.n_static)
            n_r = db.cand_assessed.n_r
            reads = 2 * n_q * S * P * T * 16 + n_q * (6 * 8 + 8 + db.batch.n_v_max * 8 + 4) + n_r * 16
            writes = n_q * db.stride * (8 + 16 + 8 + 12 + 3 * 4 * n_r + 4)
            row.update(assess_ms=kernel, assess_ms_p10_p90=[float(np.percentile(t[:, 1], 10)),
                                                             float(np.percentile(t[:, 1], 90))],
                       S=S, candidates=int((np.arange(db.stride)[None] < eng.candidate_counts(frenet, db.n_v_host)[:, None]).sum()),
                       kept_samples=int(keep.sum()), dense_tests=dense, tests_per_s=dense / (kernel * 1e-3),
                       fma_share=dense / (kernel * 1e-3) / fma_per_s, bytes_moved=reads + writes,
                       hbm_share=(reads + writes) / HBM_BYTES_PER_S / (kernel * 1e-3),
                       extra_ms_per_step=row["ms_per_step"] - plain_ms)
            hits = o["ca_dyn_hits"][..., 0]
            if S == 1:      # under the own pair the categories agree with the assessment (OK/STOP free, COLL not)
                chk = DeviceBatch(planner, frenet, bench.TARGET_SPEED, dyn_d, _lib.FOT_DYN_SINGLE, assess_candidates=True,
                                  candidate_table=True)
                chk.launch()
                cat = chk.t["cand_cat"].cpu().numpy()
                row["same_as_with_table"] = all(np.array_equal(chk.out["ca_" + k].cpu().numpy(), o["ca_" + k])
                                                for k in ("dyn_hits", "static_hit", "first_hit", "keep", "dyn_at"))
                free = (hits == 0) & (o["ca_static_hit"][..., 0] == 0)
                okstop = (cat == _lib.CAT_OK) | (cat == _lib.CAT_STOP)
                row["categories_agree"] = bool(np.all(free[okstop]) and not np.any(free[cat == _lib.CAT_COLL]))
                row["coll_candidates"] = int((cat == _lib.CAT_COLL).sum())
            else:
                live = keep > 0
                row["hit_fraction_mean"] = float(np.mean(hits[live] / S))
                row["candidates_hitting_some_sample"] = int((hits[live] > 0).sum())
        out[name] = row
    result = {"tool": "bench_assess_candidates", "card": card(), "queries": n_q, "pedestrians": int(P),
              "obstacle_steps": int(T), "n_t_max": int(eng.n_t_max), "fp64_fma_tflops": fma.value,
              "hbm_bytes_per_s": HBM_BYTES_PER_S, "variants": out}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    assert all(v["winners_unchanged"] for v in out.values()), "an assessed launch changed the winners"
    assert all(v.get("categories_agree", True) for v in out.values()), "a category disagrees with its assessment"


if __name__ == "__main__":
    main()
