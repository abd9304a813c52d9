#!/usr/bin/env python
"""bench.py -- Frenet candidate evals/s of the batched sweep (BASELINE.json metric).

One "step" = one pass of the hot path over one batch: Q independent planning queries per GPU
(SURVEY.md section 8d config 4: scenario_01 grid, 1261 candidates x 50 pedestrians x 1 sample,
51 obstacle steps), queries sharded over ranks with no data-path collective and ONE gather of the full
winner block (best_idx, best_cost, stats, winner_len, 15 winner series: 6.2 KB per query, one contiguous
buffer, one all_gather_into_tensor) per step when N > 1.

  value      dense evaluations/s with every input already resident in HBM (CUDA events, max over ranks)
  e2e        the same through the host-pointer C-ABI call `fot_plan_batch_host` (what
             FrenetPlanner.plan() binds): pinned host inputs -> H2D -> kernels -> D2H of the winners
  roofline   the sweep kernel: algorithmic 5 FLOP x evaluations / its own CUDA-event time, against the
             FP64 FMA peak measured on this GPU by fot_probe_fma_tflops (MEASURED_PEAKS.json holds no
             FP64 figure)
  cpu_baseline  the UNMODIFIED reference planner (oracle/_ref, `kind: reference`; the NumPy port when that copy
             is absent) on a bounded sample of the same queries on this box's host cores (rank 0, N = 1 only)
  parity     the reference's chosen index / cost on that sample against the GPU winners of the same queries

Weak scaling by default (Q queries per GPU); `--scaling strong` shards `--queries` over the ranks (BASELINE
config 4 as written: 4096 queries over 1/2/4/8 GPUs); at N > 1 the weak run also reports the strong figure.

`--impl reference` times only the CPU leg (all host cores) and prints the same JSON shape.

`--dump-outputs DIR` writes what the device-resident leg returned in its last timed step (rank 0's queries) as
DIR/<name>.npy, so that two builds can be compared output for output: the inputs depend only on the arguments.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests import scenarios  # noqa: E402  (seeded synthetic fields; no reference access)

METRIC = "frenet_candidate_evals_per_s"
UNIT = "evals/s"
FLOP_PER_EVAL = 5.0      # 2 SUB + 1 MUL + 1 FMA (SURVEY.md section 8d)
N_PEDS, T_OBS = 50, 51
TARGET_SPEED = 6.0
DUMP_LIMIT = 60 << 20    # array bytes --dump-outputs may write: with the file headers, under 64 MB however counted


# ------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------
def ego_and_field(qid: int):
    """Query `qid` of config 4 (seed = global query id): ego (x, y, yaw, v, a) and its pedestrian field."""
    rng = np.random.default_rng(qid)
    dyn = scenarios.pedestrian_field(rng, N_PEDS, T_OBS, scenarios.S1_KNOBS["dt"])
    ego = (rng.uniform(2, 20), rng.uniform(-1, 1), rng.normal(0, 0.05), rng.uniform(0, 8), rng.uniform(-1, 1))
    return tuple(float(v) for v in ego), dyn


def make_queries(first: int, count: int):
    """Queries first..first+count-1 of config 4: ego state -> Frenet state on the host exactly as plan()
    does it, plus that query's pedestrian field."""
    from integrated_path_planning_b200 import CubicSpline2D
    from integrated_path_planning_b200.frenet_host import CoordinateConverter, ego_to_frenet
    from integrated_path_planning_b200.types import EgoVehicleState
    spline = CubicSpline2D(*scenarios.STRAIGHT_60)
    frenet = np.empty((count, 6))
    dyn = np.empty((count, 1, N_PEDS, T_OBS, 2))
    for i in range(count):
        ego, dyn[i, 0] = ego_and_field(first + i)
        frenet[i] = ego_to_frenet(CoordinateConverter(spline), EgoVehicleState(*ego), 0.0)
    return spline, frenet, dyn


def dump_outputs(out_dir, out, query_ids):
    """The winner block `out` of queries `query_ids` as out_dir/<name>.npy in float64: best_idx, best_cost, stats,
    winner_len, winner [n, 15, n_t_max] and query_id.  Every value is finite: a query without a path (best_idx -1)
    has its infinite best_cost stored as 0, and winner samples at or past winner_len, which the kernel never writes,
    are stored as 0.  Above DUMP_LIMIT bytes a fixed, seeded sample of the queries is written."""
    host = {k: v.cpu().numpy().astype(np.float64) for k, v in out.items()}
    host["best_cost"] = np.where(host["best_idx"] >= 0, host["best_cost"], 0.0)
    host["winner"] = np.where(np.arange(host["winner"].shape[2]) < host["winner_len"][:, None, None], host["winner"], 0.0)
    host["query_id"] = np.asarray(query_ids, dtype=np.float64)
    n = len(query_ids)
    row_bytes = sum(v[0].nbytes for v in host.values())
    keep = np.arange(n)
    if n * row_bytes > DUMP_LIMIT:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), v[keep])


# ------------------------------------------------------------------------------------------
# CPU leg: the reference's own planner on the host cores
# ------------------------------------------------------------------------------------------
_CPU = {}


def _cpu_worker(qid):
    """One config-4 query through the reference's stock FrenetPlanner.plan() (or the NumPy port when oracle/_ref is
    absent).  Returns (dense evals, chosen index, cost)."""
    ego, dyn = ego_and_field(qid)
    if _CPU["kind"] == "reference":
        rec = _CPU.get("rec")
        if rec is None:
            ref = _CPU["ref"]
            pl = ref.FrenetPlanner(ref.CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
            from oracle import ref_loader
            rec = _CPU["rec"] = ref_loader.IndexRecorder(pl)
        pl = rec.planner
        pl._last_kappa = 0.0                                   # every query is an independent plan() call
        if hasattr(pl.converter, "_prev_s"):
            del pl.converter._prev_s
        path = rec.plan(_CPU["ref"].EgoVehicleState(*ego), np.empty((0, 2)), dyn, TARGET_SPEED)
        # dense credit (SURVEY.md section 8d): un-truncated samples of the grid + of the brake candidates generated
        n_c = rec.last_n_candidates
        pts = _CPU["pts_grid"] + max(0, n_c - _CPU["n_grid"]) * _CPU["n_total"] if n_c else 0
        return pts * N_PEDS, rec.last_index, (float(path.cost) if path is not None else float("inf"))
    from oracle import frenet_oracle as O
    pl = _CPU.get("port")
    if pl is None:
        pl = _CPU["port"] = O.OraclePlanner(O.Spline2D(*scenarios.STRAIGHT_60), O.Knobs(**scenarios.S1_KNOBS))
    pl.last_kappa = 0.0
    pl.search = O.NearestPointSearch(pl.sp)
    res = pl.plan(ego, np.empty((0, 2)), dyn, TARGET_SPEED)
    return int(res.n_points.sum()) * N_PEDS, res.best_index, res.cost


def cpu_setup():
    """Decide which CPU implementation runs (`reference` = unmodified copy in oracle/_ref or /root/reference)."""
    from oracle import ref_loader
    _CPU["kind"] = ref_loader.kind()
    if _CPU["kind"] == "reference":
        _CPU["ref"] = ref_loader.load()
    # dense-credit bookkeeping (SURVEY.md section 8d): samples of the un-truncated grid / brake candidates
    k = scenarios.S1_KNOBS
    n_T = int((k["max_t"] - k["min_t"]) / k["dt"] + 1e-9) + 1
    n_steps = [int(round((k["min_t"] + j * k["dt"]) / k["dt"])) + 1 for j in range(n_T)]
    n_d = 2 * int(k["max_road_width"] / k["d_road_w"] + 1e-9) + 1
    n_v = int(TARGET_SPEED / k["d_t_s"] + 1e-9) + 1
    n_v += 1 if TARGET_SPEED - (n_v - 1) * k["d_t_s"] > 1e-9 else 0
    n_total = int(round(k["max_t"] / k["dt"])) + 1
    _CPU.update(pts_grid=sum(n_steps) * n_v * n_d, n_grid=n_T * n_v * n_d, n_total=n_total)
    return _CPU["kind"]


def cpu_leg(first, n_sample, cores, steps, warmup):
    """`steps` timed passes of the CPU planner over queries first..first+n_sample-1 on a `cores`-process pool.
    Returns (evals/s, ms per pass, evals per pass, indices, costs)."""
    import multiprocessing as mp
    jobs = list(range(first, first + n_sample))
    ctx = mp.get_context("fork")           # children only run NumPy; they inherit the loaded reference modules
    with ctx.Pool(cores) as pool:
        for _ in range(warmup):
            pool.map(_cpu_worker, jobs)
        times, out = [], None
        for _ in range(steps):
            t0 = time.perf_counter()
            out = pool.map(_cpu_worker, jobs)
            times.append(time.perf_counter() - t0)
    evals = sum(o[0] for o in out)
    ms = 1e3 * float(np.mean(times))
    return evals / (ms * 1e-3), ms, evals, np.array([o[1] for o in out]), np.array([o[2] for o in out])


def cpu_plan_latency(calls=3):
    """config 2 plan() on one host core with the CPU planner: p50 in ms."""
    dyn2 = scenarios.pedestrian_field(np.random.default_rng(1), N_PEDS, T_OBS, scenarios.S1_KNOBS["dt"])
    lat = []
    if _CPU["kind"] == "reference":
        ref = _CPU["ref"]
        pl = ref.FrenetPlanner(ref.CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
        ego = ref.EgoVehicleState(5.0, 0.0, 0.0, 5.0, 0.0)
        for _ in range(calls + 1):
            pl.reset_ego_curvature()
            t0 = time.perf_counter()
            pl.plan(ego, np.empty((0, 2)), dyn2, TARGET_SPEED)
            lat.append(1e3 * (time.perf_counter() - t0))
    else:
        from oracle import frenet_oracle as O
        opl = O.OraclePlanner(O.Spline2D(*scenarios.STRAIGHT_60), O.Knobs(**scenarios.S1_KNOBS))
        for _ in range(calls + 1):
            opl.reset_ego_curvature()
            t0 = time.perf_counter()
            opl.plan((5.0, 0.0, 0.0, 5.0, 0.0), np.empty((0, 2)), dyn2, TARGET_SPEED)
            lat.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(lat[1:]))


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int, period=0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.sm, self.power, self.reasons, self.max_mhz = [], [], set(), None
        self._stop_evt = threading.Event()
        self._armed = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def arm(self):
        """Start recording (the thread and NVML are set up long before, outside any timed region)."""
        self.sm, self.power, self.reasons = [], [], set()
        self._armed.set()

    def run(self):
        if self.nv is None:
            return
        while not self._stop_evt.is_set():
            if self._armed.is_set():
                # one query per try: a box whose NVML refuses the power reading must still report clocks and reasons
                try:
                    self.sm.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                except Exception:
                    pass
                try:
                    mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    for bit, name in self.REASONS.items():
                        if mask & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
                try:
                    self.power.append(self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                except Exception:
                    pass
            time.sleep(self.period)

    def snapshot(self):
        self._armed.clear()
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "power_w": float(np.median(self.power)) if self.power else None}

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)


def _pinned_write_combined(arr):
    """A copy of `arr` in write-combined page-locked host memory (cudaHostAlloc, flag 0x04): uploads from it do not snoop
    the CPU caches.  Never freed (bench process)."""
    import ctypes as C
    rt = None
    for name in ("libcudart.so.12", "libcudart.so"):
        try:
            rt = C.CDLL(name)
            break
        except OSError:
            pass
    if rt is None:
        raise RuntimeError("libcudart not found")
    ptr = C.c_void_p()
    rc = rt.cudaHostAlloc(C.byref(ptr), C.c_size_t(arr.nbytes), C.c_uint(0x04))
    if rc != 0:
        raise RuntimeError(f"cudaHostAlloc failed: {rc}")
    buf = (C.c_char * arr.nbytes).from_address(ptr.value)
    out = np.frombuffer(buf, dtype=arr.dtype).reshape(arr.shape)
    out[...] = arr
    return out


def _ncu_traffic():
    """DRAM bytes per query of the sweep kernel and its FP64-pipe utilisation from the newest committed ncu --set full
    summary (profiles/): (bytes per query, pipe fraction, file)."""
    import glob
    import re
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*", "sweep_pairs_ncu_full_summary.txt")), reverse=True):
        txt = open(path).read()
        rd = re.search(r"dram__bytes_read\.sum\s+([\d.]+)\s*(\w*)", txt)
        wr = re.search(r"dram__bytes_write\.sum\s+([\d.]+)\s*(\w*)", txt)
        nq = re.search(r"launch__grid_size\s+(\d+)", txt)     # one CTA per query in the captured launch
        pipe = re.search(r"sm__inst_executed_pipe_fp64\.avg\.pct_of_peak_sustained_active\s+([\d.]+)", txt)
        if rd and wr and nq:
            scale = {"": 1.0, "byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            tot = float(rd.group(1)) * scale.get(rd.group(2), 1.0) + float(wr.group(1)) * scale.get(wr.group(2), 1.0)
            return tot / int(nq.group(1)), (float(pipe.group(1)) / 100.0 if pipe else None), os.path.relpath(path, ROOT)
    return None, None, None


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--queries", type=int, default=4096, help="planning queries per GPU per step (weak) / in total (strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="queries in the CPU sample (0 = 4 x cores, 2 x cores for --impl reference)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-gather", action="store_true", help="tuning: no winner gather in the timed loop")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N > 1: winners stored into the root's memory by the winner kernel over NVLink peer memory (default; "
                         "falls back to nccl when CUDA IPC is unavailable), or one all_gather_into_tensor of the packed block")
    ap.add_argument("--gather-priority", type=int, default=0, help="tuning: CUDA priority of the gather stream (0 default, -1 high)")
    ap.add_argument("--brief", action="store_true", help="resident + e2e legs only (scaling experiments)")
    ap.add_argument("--wc-input", action="store_true", help="experiment: e2e input in write-combined pinned memory (cudaHostAllocWriteCombined)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the resident leg's last-step winners (rank 0's queries) "
                                                          "as DIR/<name>.npy, float64, at most 64 MB")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = len(os.sched_getaffinity(0))
    strong = args.scaling == "strong"
    per_gpu = -(-args.queries // world) if strong else args.queries
    config = {"workload": f"config4: {'%d independent plan() queries in total' % args.queries if strong else '4096 independent plan() queries per GPU'}, "
                          "scenario_01 grid (19 d x 11 T x 6 v + 7 brake = 1261 candidates, 58041 points), "
                          "50 pedestrians x 1 sample x 51 steps, seed = query id",
              "queries_per_gpu": per_gpu, "parallelism": f"query-sharded x{world}",
              "l2": "inputs (41 KB of obstacle tracks per query, 167 MB per 4096-query step) exceed the 126 MB L2 at "
                    ">= 3100 queries per GPU; no explicit flush"}

    # ---------------- reference arm: CPU only --------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return
        kind = cpu_setup()
        n_sample = args.cpu_sample or 2 * cores
        val, ms, evals, _, _ = cpu_leg(0, n_sample, cores, args.steps, args.warmup)
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu_model(),
                                 "sample": f"each step = queries 0..{n_sample - 1} of the workload ({evals:.3g} dense evals) through "
                                           f"{'the unmodified reference FrenetPlanner.plan() (oracle/_ref)' if kind == 'reference' else 'the NumPy port'}"
                                           f", one query per task on a {cores}-process pool",
                                 "plan_p50_ms": cpu_plan_latency(),
                                 "plan_sample": "config2 plan() on one core, 3 calls after 1 warm-up"},
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ---------------- B200 arm -----------------------------------------------------------
    import torch
    import torch.distributed as dist
    from integrated_path_planning_b200 import BatchFrenetPlanner, DeviceBatch, PeerGather, WinnerBlock, _lib, shard_bounds

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the sweep has no CPU path")
    # stdout carries the one JSON line only: anything a library prints meanwhile (NCCL's version banner)
    # goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # NVML set up (tens of ms with 8 contending processes) long before any timed region
    sampler = ClockSampler(local_rank)
    sampler.start()

    if strong:
        q_lo, q_hi = shard_bounds(args.queries, world, rank)
    else:
        q_lo, q_hi = rank * args.queries, (rank + 1) * args.queries
    Q = q_hi - q_lo
    total_q = args.queries if strong else args.queries * world
    spline, frenet, dyn = make_queries(q_lo, Q)
    planner = BatchFrenetPlanner(spline, device=local_rank, **scenarios.S1_KNOBS)
    eng = planner.engine
    stream = torch.cuda.Stream(device=local_rank)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def all_max(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_list(x):
        if world == 1:
            return [float(x)]
        tk = torch.tensor([x], dtype=torch.float64, device="cuda")
        allk = torch.empty(world, dtype=torch.float64, device="cuda")
        dist.all_gather_into_tensor(allk, tk)
        return [float(v) for v in allk.cpu()]

    class ResidentLeg:
        """Inputs in HBM; per step: prepass + sweep + winner kernels and, at N > 1, the gather of the FULL winner block
        (best_idx, winner_len, stats, best_cost, 15 winner series: 6.2 KB per query), inside the timed region.

        gather = "peer" (default): the winner kernel itself stores the block a second time, into this rank's slice of a
        buffer in the ROOT's memory mapped over NVLink peer memory (PeerGather / fot_set_result_mirror) -- no collective
        call, no staging copy, nothing between two steps but the launches; the root waits on the ranks' sequence flags.
        gather = "nccl": block copied to a staging buffer, ONE all_gather_into_tensor on a side stream behind the sweep
        that produced it, N_GBUF buffers deep.  Either way the timed region ends when the last step's blocks are
        complete at their destination."""
        N_GBUF = 3

        def __init__(self, frenet, dyn, gather=True):
            self.batch = DeviceBatch(planner, frenet, TARGET_SPEED, dyn, _lib.FOT_DYN_SINGLE)
            self.mode = (args.gather if gather and world > 1 else None)
            self.step_no = 0
            self.per = int(all_max(self.batch.n_q)) if world > 1 else self.batch.n_q
            self.peer = None
            if self.mode == "peer":
                ok = 1.0
                try:
                    self.peer = PeerGather(eng, self.per, depth=self.N_GBUF)
                except Exception as exc:                     # CUDA IPC not available in this container: one rank fails, all fall back
                    print(f"[bench] rank {rank}: peer gather unavailable ({exc!r}); falling back to nccl", file=sys.stderr)
                    ok = 0.0
                if all_max(1.0 - ok) > 0.0:
                    if self.peer is not None:
                        self.peer.close()
                    self.peer, self.mode = None, "nccl"
            if self.mode == "nccl":
                self.gstream = torch.cuda.Stream(device=local_rank, priority=args.gather_priority)
                self.stage = [WinnerBlock(self.per, eng.n_t_max, device="cuda") for _ in range(self.N_GBUF)]
                for s in self.stage:
                    s.buf.zero_()
                self.gathered = [torch.empty((world, self.stage[0].nbytes), dtype=torch.uint8, device="cuda")
                                 for _ in range(self.N_GBUF)]
                self.g_done = [None] * self.N_GBUF
            self.gather = self.mode is not None
            self.n_mirrored = 0

        def step(self):
            if self.mode == "peer":
                self.peer.attach(self.step_no)               # this launch's winners also go to buffer step_no % depth on the root
                self.batch.launch(stream.cuda_stream)
                self.step_no += 1
                self.n_mirrored += 1
                return
            self.batch.launch(stream.cuda_stream)
            if self.mode != "nccl":
                return
            k = self.step_no % self.N_GBUF
            self.step_no += 1
            with torch.cuda.stream(stream):
                if self.g_done[k] is not None:
                    stream.wait_event(self.g_done[k])            # the gather that last read this staging buffer
                if self.per == self.batch.n_q:
                    self.stage[k].buf.copy_(self.batch.block.buf, non_blocking=True)
                else:                                            # uneven shards: section by section into the padded block
                    for key, v in self.batch.out.items():
                        self.stage[k].views[key][:self.batch.n_q].copy_(v, non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(stream)
            with torch.cuda.stream(self.gstream):
                self.gstream.wait_event(ready)
                dist.all_gather_into_tensor(self.gathered[k].view(-1), self.stage[k].buf)
                self.g_done[k] = torch.cuda.Event()
                self.g_done[k].record(self.gstream)

        def run(self, steps, warmup):
            for _ in range(warmup):
                self.step()
            sync_all()
            sampler.arm()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                if world > 1:
                    # ranks aligned ON THE DEVICE: a collective on the timing stream right before the start event
                    dist.all_reduce(torch.zeros(1, device="cuda"))
                e0.record()
            for _ in range(steps):
                self.step()
            with torch.cuda.stream(stream):
                if self.mode == "nccl":
                    stream.wait_stream(self.gstream)             # the timed region ends after the last gather
                if self.mode == "peer" and rank == self.peer.root:
                    # ... on the root: after every rank's last block has arrived (device-side wait on the sequence flags)
                    self.peer.await_step(self.n_mirrored, stream.cuda_stream)
                e1.record()
            sync_all()
            clocks = sampler.snapshot()
            n_timed = min(steps, 256)
            stage = np.array([eng.launch_stage_ms(b) for b in range(n_timed)])   # [prepass, sweep, winner]
            return all_max(e0.elapsed_time(e1)) / steps, stage, clocks

        def verify_gather(self):
            """The last step's gathered blocks, slice by slice, against what each rank computed itself."""
            if not self.gather:
                return None
            n = self.batch.n_q
            k = (self.step_no - 1) % self.N_GBUF
            # every rank's own (best_idx, winner_len, stats) checksum and cost bits, gathered the plain way
            def digest(o, c):
                # (winner rows are written up to winner_len only: the first two x samples count where a path exists)
                head = torch.where((o["winner_len"][:c] >= 2)[:, None], o["winner"][:c, 9, :2], 0.0)
                return torch.stack([o["best_idx"][:c].to(torch.int64).sum(), o["winner_len"][:c].to(torch.int64).sum(),
                                    o["stats"][:c].to(torch.int64).sum(), o["best_cost"][:c].contiguous().view(torch.int64).sum(),
                                    head.contiguous().view(torch.int64).sum()])
            own = digest(self.batch.out, n)
            all_own = torch.empty((world, 5), dtype=torch.int64, device="cuda")
            dist.all_gather_into_tensor(all_own.view(-1), own)
            ok = True
            if self.mode == "peer":
                if rank == self.peer.root:
                    ok = not self.peer.timed_out()
                    got = self.peer.views(self.step_no - 1)
            else:
                got = self.stage[k].unpack(self.gathered[k])
            if self.mode == "nccl" or rank == self.peer.root:
                counts = [int(c) for c in all_list(n)]
                for r in range(world):
                    c = counts[r]
                    seen = digest({key: v[r] for key, v in got.items()}, c)
                    ok = ok and bool(torch.equal(seen, all_own[r]))
                mine = got["winner"][rank, :n]
                lens = self.batch.out["winner_len"]
                keep = torch.arange(mine.shape[-1], device="cuda")[None, None, :] < lens[:, None, None]
                ok = ok and bool(torch.equal(torch.where(keep, mine, 0.0).view(torch.int64),
                                             torch.where(keep, self.batch.out["winner"], 0.0).view(torch.int64)))
            else:
                all_list(n)
            return bool(all_max(0.0 if ok else 1.0) == 0.0)

        def close(self):
            if self.peer is not None:
                sync_all()
                self.peer.close()
                self.peer = None

    leg = ResidentLeg(frenet, dyn, gather=not args.no_gather)
    evals_local = leg.batch.dense_evals()
    evals_total = float(sum(all_list(evals_local)))
    ms_step, stage, clocks = leg.run(args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, leg.batch.out, np.arange(q_lo, q_hi))
    gather_ok = leg.verify_gather()
    sweep_ms = float(stage[:, 1].mean())
    value = evals_total / (ms_step * 1e-3)
    per_rank_ms = all_list(float(stage.sum(axis=1).mean()))
    per_rank_mhz = all_list(float(clocks.get("sm_mhz") or 0.0))
    per_rank_w = all_list(float(clocks.get("power_w") or 0.0))
    gather_bytes = WinnerBlock(leg.per, eng.n_t_max, device="meta").nbytes if leg.gather else 0
    gather_mode = leg.mode
    leg.close()
    resident_best = leg.batch.out["best_idx"].cpu().numpy()
    resident_cost = leg.batch.out["best_cost"].cpu().numpy()

    # the other scaling mode, same run (N > 1 only): BASELINE config 4 as written = 4096 queries in total
    other = None
    if world > 1 and not args.brief:
        if strong:
            o_lo, o_hi, o_total = rank * args.queries, (rank + 1) * args.queries, args.queries * world
        else:
            o_lo, o_hi = shard_bounds(args.queries, world, rank)
            o_total = args.queries
        _, fr_o, dyn_o = make_queries(o_lo, o_hi - o_lo) if (o_lo, o_hi) != (q_lo, q_hi) else (None, frenet, dyn)
        leg_o = ResidentLeg(fr_o, dyn_o, gather=not args.no_gather)
        ev_o = float(sum(all_list(leg_o.batch.dense_evals())))
        ms_o, stage_o, _ = leg_o.run(max(args.steps, 20), args.warmup)
        other = {"scaling": "weak" if strong else "strong", "queries_total": o_total, "queries_per_gpu": o_hi - o_lo,
                 "value": ev_o / (ms_o * 1e-3), "unit": UNIT, "ms_per_step": ms_o,
                 "per_rank_kernel_ms_per_step": all_list(float(stage_o.sum(axis=1).mean())),
                 "gather_ok": leg_o.verify_gather()}
        leg_o.close()
        del leg_o

    # e2e leg: host-pointer C-ABI call, pinned inputs, H2D + kernels + D2H inside the timed region
    if args.wc_input:
        dyn_host = _pinned_write_combined(dyn)                # experiment: write-combined page-locked input (no snooping on the upload)
    else:
        dyn_pinned = torch.from_numpy(dyn).pin_memory()
        dyn_host = dyn_pinned.numpy()
    for _ in range(args.warmup):
        res = planner.plan_batch(frenet, TARGET_SPEED, dynamic_obstacles=dyn_host[:, 0])
    e2e_steps = args.steps
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        res = planner.plan_batch(frenet, TARGET_SPEED, dynamic_obstacles=dyn_host[:, 0])
    if world > 1:
        dist.barrier()
    e2e_ms = all_max(1e3 * (time.perf_counter() - t0) / e2e_steps)
    h2d = dyn.nbytes + frenet.nbytes + Q * (8 + 32 + 8 + 4) + Q * 6 * 8
    d2h = res.best_idx.nbytes + res.best_cost.nbytes + res.stats.nbytes + res.winner_len.nbytes + res.winner.nbytes
    # resident and e2e legs must pick the same winners
    same = bool(np.array_equal(resident_best, res.best_idx))
    e2e_best = res.best_idx.copy()
    cand_total = float(sum(all_list(float(res.n_cand.sum()))))

    e2e_cv = None
    if not args.brief:
        # e2e with the predictor's post-processing on the device (SURVEY.md section 8f, rank 1): the caller hands
        # over the last two pedestrian observations and the current positions (host, pinned) instead of the
        # obstacle tensor; constant-velocity extrapolation + t = 0 column are built on the GPU and feed the sweep.
        from integrated_path_planning_b200.prediction import DevicePredictionPostprocessor
        post = DevicePredictionPostprocessor(pred_len=12, sgan_dt=0.4, sim_dt=scenarios.S1_KNOBS["dt"], plan_horizon=5.0,
                                             device=local_rank)
        p0 = dyn[:, 0, :, 0, :]
        vel = (dyn[:, 0, :, 1, :] - dyn[:, 0, :, 0, :]) / scenarios.S1_KNOBS["dt"]
        host_in = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (p0, p0 - vel * 0.4, p0)]
        dev_in = [torch.empty_like(a, device="cuda") for a in host_in]
        dyn_buf = torch.empty((Q, 1, N_PEDS, post.n_steps + 1, 2), dtype=torch.float64, device="cuda")
        batch_cv = DeviceBatch(planner, frenet, TARGET_SPEED, dyn_buf, _lib.FOT_DYN_SINGLE)
        host_out = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in batch_cv.out.items()}

        def cv_step():
            with torch.cuda.stream(stream):
                for d, h_ in zip(dev_in, host_in):
                    d.copy_(h_, non_blocking=True)
                post.predict_cv(dev_in[0], dev_in[1], None, dev_in[2], out=dyn_buf)
            batch_cv.launch_to_host(host_out, stream.cuda_stream)    # ranges of queries; winners go back while the rest is swept

        for _ in range(args.warmup):
            cv_step()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            cv_step()
        if world > 1:
            dist.barrier()
        cv_ms = all_max(1e3 * (time.perf_counter() - t0) / e2e_steps)
        cv_match = float(np.mean(host_out["best_idx"].numpy() == e2e_best))
        # the same route with the compact read-back (first two samples of every winner series: what a closed-loop caller
        # consumes): the variant that does not depend on the host's PCIe path at 8 GPUs
        K_HEAD = 2
        host_out_c = {k: (torch.empty((Q, v.shape[1], K_HEAD), dtype=v.dtype) if k == "winner" else torch.empty(v.shape, dtype=v.dtype)).pin_memory()
                      for k, v in batch_cv.out.items()}

        def cv_step_compact():
            with torch.cuda.stream(stream):
                for d, h_ in zip(dev_in, host_in):
                    d.copy_(h_, non_blocking=True)
                post.predict_cv(dev_in[0], dev_in[1], None, dev_in[2], out=dyn_buf)
            batch_cv.launch_to_host(host_out_c, stream.cuda_stream, winner_samples=K_HEAD)

        for _ in range(args.warmup):
            cv_step_compact()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            cv_step_compact()
        if world > 1:
            dist.barrier()
        cvc_ms = all_max(1e3 * (time.perf_counter() - t0) / e2e_steps)
        has_path = host_out["best_idx"].numpy() >= 0
        heads_ok = bool(np.array_equal(host_out_c["best_idx"].numpy(), host_out["best_idx"].numpy()) and
                        np.array_equal(host_out_c["winner"].numpy()[has_path], host_out["winner"].numpy()[has_path][:, :, :K_HEAD]))
        e2e_cv_compact = {"value": evals_total / (cvc_ms * 1e-3), "unit": UNIT, "ms_per_step": cvc_ms, "winner_samples": K_HEAD,
                          "h2d_bytes_per_step": int(sum(a.numel() * 8 for a in host_in)),
                          "d2h_bytes_per_step": int(sum(v.numel() * v.element_size() for v in host_out_c.values())),
                          "equal_to_full_read_back": heads_ok}
        e2e_cv = {"value": evals_total / (cv_ms * 1e-3), "unit": UNIT, "ms_per_step": cv_ms, "compact": e2e_cv_compact,
                  "h2d_bytes_per_step": int(sum(a.numel() * 8 for a in host_in)),
                  "d2h_bytes_per_step": int(sum(v.numel() * v.element_size() for v in host_out.values())),
                  "winners_equal_to_tensor_path": cv_match,
                  "note": "inputs = last two observations + current positions per query (host, pinned); constant-velocity "
                          "obstacle tensor built on the device (fot_predict_cv_device), then the same sweep"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        sampler.stop()
        return

    # FP64 pipe peak measured here (2 FLOP per FMA)
    import ctypes as C
    peak = C.c_double()
    _lib.check(eng.lib.fot_probe_fma_tflops(local_rank, 0, C.byref(peak)), "probe")
    achieved_tf = FLOP_PER_EVAL * evals_local / (sweep_ms * 1e-3) / 1e12
    per_q, pipe_util, src = _ncu_traffic()
    roofline = {"bound": "fp64_pipe", "achieved": achieved_tf, "peak": peak.value, "unit": "TFLOP/s",
                "frac": achieved_tf / peak.value,
                "traffic": per_q * Q if per_q else None,
                "traffic_source": f"constant from {src} (ncu --set full, dram read + write bytes per query x queries); not measured in this run" if src else None,
                "pipe_util_ncu": pipe_util,
                "pipe_util_note": f"sm__inst_executed_pipe_fp64 of the same kernel and workload, constant from {src}: the FP64 pipe's own busy "
                                  "fraction, next to the dense-credit `frac` (which counts every candidate x obstacle x step test, "
                                  "most of which the kernel culls -- it can exceed 1)" if src else None,
                "kernel": {4: "fot_sweep_pairs", 1: "fot_sweep_items", 3: "fot_sweep_warp", 2: "fot_sweep"}.get(
                    int(eng.lib.fot_last_sweep_kind(eng._h)), "?"), "kernel_ms": sweep_ms,
                "stage_ms": {"prepass": float(stage[:, 0].mean()), "sweep": sweep_ms, "winner": float(stage[:, 2].mean())},
                "peak_source": "fot_probe_fma_tflops on this GPU (dependent-chain DFMA, 2 FLOP/FMA); "
                               "MEASURED_PEAKS.json has no FP64 figure",
                "note": "algorithmic 5 FLOP per dense evaluation (dense credit: the kernel culls, so this is not pipe "
                        "utilisation -- ncu's sm__inst_executed_pipe_fp64 is in profiles/); point generation (about 58041 "
                        "points per query) is extra work not credited here"}

    plan_latency = closed_loop = None
    if not args.brief:
        # plan() latency (BASELINE config 2: one call, default grid, 50 pedestrians x 1 sample), measured the
        # way the reference's simulator measures it: time.perf_counter around FrenetPlanner.plan()
        # (integrated_simulator.py:575-585) -- ego->Frenet on the host, H2D, kernels, D2H, FrenetPath rebuilt
        from integrated_path_planning_b200 import FrenetPlanner
        from integrated_path_planning_b200.types import EgoVehicleState
        single = FrenetPlanner(spline, device=local_rank, **scenarios.S1_KNOBS)
        ego2 = EgoVehicleState(x=5.0, y=0.0, yaw=0.0, v=5.0, a=0.0)
        dyn2 = scenarios.pedestrian_field(np.random.default_rng(1), N_PEDS, T_OBS, scenarios.S1_KNOBS["dt"])
        lat, kms = [], []
        for i in range(103):
            single.reset_ego_curvature()
            t0 = time.perf_counter()
            single.plan(ego2, np.empty((0, 2)), dyn2, TARGET_SPEED)
            lat.append(1e3 * (time.perf_counter() - t0))
            kms.append(single.last_result.kernel_ms)
        plan_latency = {"p50_ms": float(np.median(lat[3:])), "p95_ms": float(np.percentile(lat[3:], 95)),
                        "kernels_p50_ms": float(np.median(kms[3:])), "calls": 100,
                        "config": "config2: one plan() call, 1261 candidates x 50 pedestrians x 1 sample"}

        # closed-loop campaign (SURVEY.md section 8f, rank 3): 256 simulations of the recorded scenario_01 variants (with
        # jitter) advanced in lock-step by the batched driver; informational, never allowed to break the bench line
        try:
            golden = os.path.join(ROOT, "tests", "golden", "rollout_s01.npz")
            if world == 1 and os.path.exists(golden):
                from integrated_path_planning_b200.rollout import BatchedClosedLoop
                z = np.load(golden)
                knobs = {k[5:]: float(z[k]) for k in z.files if k.startswith("knob/")}
                rng_cl = np.random.default_rng(7)
                n_sims, n_var = 256, int(z["n_variants"])
                tracks = np.stack([z[f"v{i % n_var}/traj"] + rng_cl.normal(0.0, 0.3, (1, z["v0/traj"].shape[1], 2)) for i in range(n_sims)])
                ego0 = np.stack([z[f"v{i % n_var}/ego0"] for i in range(n_sims)])
                sim = BatchedClosedLoop(z["v0/wx"], z["v0/wy"], knobs, tracks, ego0, device=local_rank)
                sim.warmup()
                for _ in range(3):
                    sim.step()
                calls0, t0, sim_steps = sim.n_plan_calls, time.perf_counter(), 0
                for _ in range(30):
                    sim_steps += int(sim.active.sum())
                    sim.step()
                wall = time.perf_counter() - t0
                closed_loop = {"sim_steps_per_s": sim_steps / wall, "plan_calls_per_s": (sim.n_plan_calls - calls0) / wall,
                               "sims": n_sims, "lockstep_ms": 1e3 * wall / 30,
                               "note": "BatchedClosedLoop: observer, CV prediction, safety metrics, fail-safe state machine, sweep "
                                       "(+ escalation retries), ego update per step; the reference runs ~4.8 such steps/s"}
        except Exception as exc:                     # pragma: no cover
            closed_loop = {"error": repr(exc)}

    cpu = parity = None
    if world == 1 and not args.no_cpu and not args.brief:
        kind = cpu_setup()
        n_sample = min(Q, args.cpu_sample or 4 * cores)
        val, ms, ev, cpu_idx, cpu_cost = cpu_leg(q_lo, n_sample, cores, 2, 1)
        cpu = {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu_model(),
               "sample": f"queries 0..{n_sample - 1} of the {Q} ({ev:.3g} dense evals) through "
                         f"{'the unmodified reference FrenetPlanner.plan() (oracle/_ref)' if kind == 'reference' else 'the NumPy port'}"
                         f" on a {cores}-process pool, mean of 2 passes after 1 warm-up, {ms:.0f} ms per pass",
               "plan_p50_ms": cpu_plan_latency(),
               "plan_sample": "config2 plan() on one core, 3 calls after 1 warm-up"}
        # parity of the timed workload: the CPU planner's choice against the GPU winners of the same queries
        gi, gc = resident_best[:n_sample], resident_cost[:n_sample]
        found = cpu_idx >= 0
        rel = np.abs(gc[found & (gi >= 0)] - cpu_cost[found & (gi >= 0)]) / np.abs(cpu_cost[found & (gi >= 0)])
        parity = {"queries": int(n_sample), "index_mismatches": int(np.sum(gi != cpu_idx)),
                  "e2e_index_mismatches": int(np.sum(e2e_best[:n_sample] != cpu_idx)),
                  "with_a_path": int(found.sum()), "max_rel_cost": float(rel.max()) if rel.size else 0.0,
                  "against": kind}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config, "clocks": clocks,
            "e2e": {"value": evals_total / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms, "steps": e2e_steps,
                    "winners_match_resident": same},
            "gpu_launches": 4 * args.steps, "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
            "gather": {"bytes_per_rank_per_step": int(gather_bytes), "mode": gather_mode,
                       "collectives_per_step": 1 if gather_mode == "nccl" else 0,
                       "what": "full winner block (best_idx, winner_len, stats, best_cost, 15 winner series) of every rank, inside "
                               "the timed region: " + ("stored into the root's memory by each rank's winner kernel over NVLink peer "
                               "memory (fot_set_result_mirror), sequence flags awaited on the root" if gather_mode == "peer" else
                               "one contiguous buffer, one all_gather_into_tensor"),
                       "verified": gather_ok} if world > 1 else None,
            "per_rank_kernel_ms_per_step": per_rank_ms, "per_rank_sm_mhz": per_rank_mhz, "per_rank_power_w": per_rank_w,
            "other_scaling": other,
            "plan_latency": plan_latency, "e2e_device_prediction": e2e_cv, "closed_loop": closed_loop,
            "candidates_per_s": cand_total / (ms_step * 1e-3),
            "evals_per_step_per_gpu": evals_local, "queries_total": total_q}
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    os.dup2(2, 1)
    sampler.stop()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
