"""End-to-end (host-pointer C-ABI) timing of the bench workload only: python tools/tuning/e2e_probe.py [queries] [reps]
Environment knobs (FOT_HOST_CHUNKS, ...) are resolved per handle; PROBE_VARIANTS switches them with reload_options()."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np, torch
import bench
from tests import scenarios
from integrated_path_planning_b200 import BatchFrenetPlanner
nq = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 12
spline, frenet, dyn = bench.make_queries(0, nq)
planner = BatchFrenetPlanner(spline, device=0, **scenarios.S1_KNOBS)
dyn_host = dyn if os.environ.get("PROBE_PAGEABLE") else torch.from_numpy(dyn).pin_memory().numpy()   # PROBE_PAGEABLE=1: an ordinary NumPy array
variants = [v for v in os.environ.get("PROBE_VARIANTS", "").split(";") if v] or [""]
ref = None
for v in variants:
    for kv in v.split():
        k, val = kv.split("=")
        os.environ[k] = val
    planner.engine.reload_options()
    for _ in range(4):
        res = planner.plan_batch(frenet, bench.TARGET_SPEED, dynamic_obstacles=dyn_host[:, 0])
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = planner.plan_batch(frenet, bench.TARGET_SPEED, dynamic_obstacles=dyn_host[:, 0])
        ts.append(1e3 * (time.perf_counter() - t0))
    if ref is None:
        ref = res.best_idx.copy()
    same = bool(np.array_equal(ref, res.best_idx))
    print(f"{v or 'default':60s} median {np.median(ts):.3f} ms  min {min(ts):.3f}  same_winners {same}", flush=True)
    for kv in v.split():
        os.environ.pop(kv.split("=")[0], None)
    planner.engine.reload_options()
