#!/usr/bin/env python
"""Cost-weight sweeps: what selecting every query's winner under n_w weightings costs on top of a resident config-4
launch, against the separate sweeps it replaces.

    python tools/bench_weights.py --queries 4096 --steps 100 --warmup 5 --out profiles/r3/bench_weights.json

The config-4 queries of bench.py (4096 resident queries, 50 pedestrians each) go through `DeviceBatch` in variants
that alternate in one process: the plain launch (what bench.py times); cost_weights with n_w = 1 / 8 / 64 / 256
without series; n_w = 8 with series; cost_terms alone; and `separate8`, eight plain launches on eight handles built
with the same eight weightings -- the way to get the same answers without this feature.  Every step is timed with
CUDA events on one stream: `sweep_ms` is the fot_plan_batch_device launch, `extra_ms` what follows it
(fot_select_weighted, fot_cost_terms), `ms_per_step` both.  After the timed steps the n_w = 8 selections (index, cost
bits, length, series bits) must equal the eight separate sweeps, and every weighted variant's first weighting (the
handle's own) must equal its own winner.  Then one 256-simulation roll-out is stepped with and without cost_weights
(each simulation its own weighting) and the lock-step time is reported.  Prints one JSON line with the card's name and
power limit, read in the same run.
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

KEYS = ("k_j", "k_t", "k_d", "k_s_dot", "k_lat", "k_lon")


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def weightings(own, n, seed=11):
    """n weightings: the handle's own first, then log-uniform factors of 1e-2 .. 1e2 on each knob."""
    rng = np.random.default_rng(seed)
    w = own[None] * 10.0 ** rng.uniform(-2.0, 2.0, size=(n, 6))
    w[0] = own
    return w


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def check_against_separate(db, separate):
    """Index, cost bits, kept length and series bits of every selection equal the sweep of the handle with that
    weighting."""
    o = {k: v.cpu().numpy() for k, v in db.out.items()}
    ok = True
    for w, sb in enumerate(separate):
        s = {k: v.cpu().numpy() for k, v in sb.out.items()}
        ok &= np.array_equal(o["w_idx"][:, w], s["best_idx"])
        ok &= np.array_equal(bits(o["w_cost"][:, w]), bits(s["best_cost"]))
        rows = np.nonzero(s["best_idx"] >= 0)[0]
        ok &= np.array_equal(o["w_len"][rows, w], s["winner_len"][rows])
        live = np.arange(s["winner"].shape[-1])[None, None, :] < s["winner_len"][rows].reshape(-1, 1, 1)
        ok &= np.array_equal(bits(np.where(live, o["w_series"][rows, w], 0.0)), bits(np.where(live, s["winner"][rows], 0.0)))
    return bool(ok)


def check_own(db):
    o = {k: v.cpu().numpy() for k, v in db.out.items()}
    return bool(np.array_equal(o["w_idx"][:, 0], o["best_idx"]) and np.array_equal(bits(o["w_cost"][:, 0]), bits(o["best_cost"])))


def rollout_ms(sims, steps, weighted):
    """ms per lock-step of tools/bench_rollout.py's campaign (scenario_01 variants tiled to `sims`, seeded jitter),
    with a weighting per simulation when `weighted`."""
    from integrated_path_planning_b200.rollout import BatchedClosedLoop
    z = np.load(os.path.join(ROOT, "tests", "golden", "rollout_s01.npz"))
    knobs = {k[5:]: float(z[k]) for k in z.files if k.startswith("knob/")}
    rng = np.random.default_rng(7)
    n_var = int(z["n_variants"])
    tracks, ego0 = [], []
    for i in range(sims):
        v = i % n_var
        t = z[f"v{v}/traj"]
        tracks.append(t + rng.normal(0.0, 0.3, (1, t.shape[1], 2)))
        e = z[f"v{v}/ego0"].copy()
        e[3] = max(0.5, e[3] + rng.normal(0.0, 0.3))
        ego0.append(e)
    cw = weightings(np.array([knobs[k] for k in KEYS]), sims, seed=3) if weighted else None
    sim = BatchedClosedLoop(z["v0/wx"], z["v0/wy"], knobs, np.stack(tracks), np.stack(ego0), cost_weights=cw)
    sim.warmup()
    for _ in range(3):
        sim.step()
    t0 = time.perf_counter()
    for _ in range(steps):
        sim.step()
    return 1e3 * (time.perf_counter() - t0) / steps, int(sim.active.sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=100, help="timed steps per variant, in rounds of --block")
    ap.add_argument("--block", type=int, default=20, help="consecutive steps of one variant before the next one runs")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rollout-sims", type=int, default=256)
    ap.add_argument("--rollout-steps", type=int, default=60)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    import bench
    from tests import scenarios
    from integrated_path_planning_b200 import _lib
    from integrated_path_planning_b200.batch import BatchFrenetPlanner, DeviceBatch
    from integrated_path_planning_b200 import CubicSpline2D
    if not torch.cuda.is_available():
        raise SystemExit("bench_weights.py needs a CUDA device")
    planner = BatchFrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    own = np.array([float(scenarios.S1_KNOBS[k]) for k in KEYS])
    w8 = weightings(own, 8)
    _, frenet, dyn = bench.make_queries(0, args.queries)
    dyn_d = torch.from_numpy(dyn).cuda()
    mk = lambda pl, **kw: DeviceBatch(pl, frenet, bench.TARGET_SPEED, dyn_d, _lib.FOT_DYN_SINGLE, **kw)
    batches = {"plain": mk(planner)}
    for n_w in (1, 8, 64, 256):
        batches[f"w{n_w}"] = mk(planner, cost_weights=weightings(own, n_w), weight_series=False)
    batches["w8_series"] = mk(planner, cost_weights=w8)
    batches["cost_terms"] = mk(planner, cost_terms=True)
    separate = [mk(BatchFrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **dict(scenarios.S1_KNOBS, **dict(zip(KEYS, w)))))
                for w in w8]
    names = list(batches) + ["separate8"]
    stream = torch.cuda.Stream()
    raw = stream.cuda_stream
    eng = planner.engine

    def step(name, ev):
        ev[0].record(stream)
        if name == "separate8":
            for sb in separate:
                sb.engine.run_device(sb.batch, sb.result, raw)
            ev[1].record(stream)
        else:
            db = batches[name]
            eng.run_device(db.batch, db.result, raw)
            ev[1].record(stream)
            if db.n_w > 0:
                eng.select_weighted_device(db.batch, db.result.cand_cat, db.stride, db.weighted, raw)
            if db.cost_terms:
                eng.cost_terms_device(db.batch, db.stride, db.out["cost_terms"].data_ptr(), raw)
        ev[2].record(stream)

    new_ev = lambda: [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    with torch.cuda.stream(stream):
        for name in names:
            for _ in range(args.warmup):
                step(name, new_ev())
        stream.synchronize()
        times = {name: [] for name in names}
        for _ in range(max(1, -(-args.steps // args.block))):
            for name in names:
                evs = [new_ev() for _ in range(args.block)]
                for ev in evs:
                    step(name, ev)
                stream.synchronize()
                times[name] += [(ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[0].elapsed_time(ev[2]))
                                for ev in evs]
    out = {}
    for name in names:
        t = np.array(times[name])
        row = {"steps": len(t), "ms_per_step": float(np.median(t[:, 2])), "sweep_ms": float(np.median(t[:, 0])),
               "extra_ms": float(np.median(t[:, 1])),
               "ms_per_step_p10_p90": [float(np.percentile(t[:, 2], 10)), float(np.percentile(t[:, 2], 90))]}
        db = batches.get(name)
        if db is not None and db.n_w > 0:
            row["n_w"] = db.n_w
            row["series"] = "w_series" in db.out
            row["own_weighting_is_the_winner"] = check_own(db)
        out[name] = row
    identical = check_against_separate(batches["w8_series"], separate)
    n_q = args.queries
    stride = int(batches["plain"].stride)
    r_plain, act_plain = rollout_ms(args.rollout_sims, args.rollout_steps, False)
    r_w, act_w = rollout_ms(args.rollout_sims, args.rollout_steps, True)
    result = {"tool": "bench_weights", "card": card(), "queries": n_q, "candidates_per_query": stride,
              "cost_evaluations_per_weighting": n_q * stride, "fp64_ops_per_weighting": 13 * n_q * stride,
              "selection_bit_identical_to_8_separate_sweeps": identical, "variants": out,
              "rollout": {"sims": args.rollout_sims, "steps": args.rollout_steps,
                          "ms_per_lockstep_plain": r_plain, "ms_per_lockstep_cost_weights": r_w,
                          "still_active": [act_plain, act_w]}}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    assert identical, "weighted selection differs from the separate sweeps"
    assert all(v.get("own_weighting_is_the_winner", True) for v in out.values()), "own weighting != winner"


if __name__ == "__main__":
    main()
