"""The nearest-point search on the device (fot_nearest_s_device) behind BatchCoordinateConverter(engine=...) and
BatchFrenetPlanner.plan_batch_from_ego: bit for bit what the host computes, through cached windows, stale windows,
first calls, path ends and near ties, and certified on the device for nearly every row (DESIGN.md section 4e).
Every comparison is exact (np.array_equal), never a tolerance."""
import math
import os
import subprocess

import numpy as np
import pytest

from integrated_path_planning_b200.frenet_host import (BatchCoordinateConverter, CoordinateConverter, ego_to_frenet,
                                                       ego_to_frenet_many)
from integrated_path_planning_b200.spline import CubicSpline2D, spline_tables
from integrated_path_planning_b200.types import EgoVehicleState
from tests import runners, scenarios
from tests.test_batch_converter import _curved_path, _path, _walks

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CUBE_ULPS = 4            # kCubeUlps of csrc/fot_frenet.cuh


def _s_curve():
    """A long S-curve with 61 knots: more than the 48 that fot_sweep_pairs keeps in shared memory."""
    s = np.linspace(0.0, 300.0, 61)
    return CubicSpline2D(list(s), list(15.0 * np.sin(s / 20.0)))


PATHS = {"straight": _path, "curved": _curved_path, "s_curve": _s_curve}
_ENGINES = {}


def _engine(name):
    """One planner (and device handle) per test path."""
    if name not in _ENGINES:
        from integrated_path_planning_b200.batch import BatchFrenetPlanner
        _ENGINES[name] = BatchFrenetPlanner(PATHS[name]())
    return _ENGINES[name].engine


def _past_the_ends(path, ego, rng):
    """Move a few egos beyond either end of the path, along the end tangents."""
    out = ego.copy()
    length = path.s[-1]
    for k in np.nonzero(rng.random(len(ego)) < 0.05)[0]:
        at_end = rng.random() < 0.5
        s = length if at_end else 0.0
        px, py = path.calc_position(s)
        yaw = float(path.calc_yaw(s))
        reach = rng.uniform(0.5, 15.0) * (1.0 if at_end else -1.0)
        out[k, 0] = float(px) + reach * math.cos(yaw)
        out[k, 1] = float(py) + reach * math.sin(yaw) + rng.normal(0.0, 1.0)
    return out


_SHARE = {}


@pytest.mark.parametrize("name", sorted(PATHS))
def test_random_walks_equal_the_scalar_converter(name):
    """(a) Changing subsets, jumps that make the window stale, first calls, egos past both ends: Frenet states, ok and
    the caches equal N scalar CoordinateConverters after every call."""
    path = PATHS[name]()
    rng = np.random.default_rng({"straight": 11, "curved": 12, "s_curve": 13}[name])
    n, steps = 48, 60
    ego = _walks(path, n, steps, rng)
    kappa = rng.normal(0, 0.05, (steps, n))
    scalar = [CoordinateConverter(path) for _ in range(n)]
    dev = BatchCoordinateConverter(path, n, engine=_engine(name))
    for t in range(steps):
        idx = np.nonzero(rng.random(n) < 0.8)[0]
        if len(idx) == 0:
            continue
        e = _past_the_ends(path, ego[t, idx], rng)
        got, ok = ego_to_frenet_many(dev, idx, e, kappa[t, idx])
        for j, i in enumerate(idx):
            want = ego_to_frenet(scalar[i], EgoVehicleState(*e[j]), float(kappa[t, i]))
            assert ok[j] == (want is not None), (t, i)
            if want is not None:
                assert np.array_equal(got[j], want), (t, i, got[j] - want)
            assert np.array_equal(dev.prev_s[i], getattr(scalar[i], "_prev_s", np.nan), equal_nan=True), (t, i)
    assert dev.device_rows + dev.host_rows > 0
    _SHARE[name] = (dev.device_rows, dev.host_rows)


def test_near_tie_goes_back_to_the_host():
    """(b) The bisector point of two window samples: the device cannot certify the window's arg-min, reports
    status 1, and the host answers with the reference's arithmetic."""
    path = _path()
    grid = np.linspace(0.0, 20.0, 100)
    mid = 0.5 * (grid[40] + grid[41])
    px, py = path.calc_position(mid)
    x, y = float(np.asarray(px).reshape(-1)[0]), float(np.asarray(py).reshape(-1)[0]) + 0.7
    eng = _engine("straight")
    _, status = eng.nearest_s(np.array([x]), np.array([y]), np.array([10.0]))
    assert status[0] == 1
    scalar = CoordinateConverter(path)
    scalar._prev_s = 10.0
    want = scalar.find_nearest_point_on_path(x, y)[0]
    dev = BatchCoordinateConverter(path, 1, engine=eng)
    dev.prev_s[0] = 10.0
    got = dev.nearest_s([0], [x], [y])[0]
    assert dev.host_rows == 1 and dev.device_rows == 0
    assert got == want and dev.prev_s[0] == scalar._prev_s


def test_unusual_inputs_go_back_to_the_host():
    """NaN or infinite positions and caches, a cache past the path end: status 1, and the converter returns what the
    host converter returns (a NaN position is no conversion failure in the reference: it gives a NaN Frenet state)."""
    path = _path()
    eng = _engine("straight")
    end = float(path.s[-1])
    x = np.array([np.nan, 5.0, np.inf, 5.0, 5.0, 5.0])
    y = np.array([0.5, np.nan, 0.5, 0.5, 0.5, 0.5])
    prev = np.array([np.nan, 3.0, np.nan, np.inf, -np.inf, end + 50.0])
    _, status = eng.nearest_s(x, y, prev)
    assert (status == 1).all()
    ego = np.zeros((len(x), 5))
    ego[:, 0], ego[:, 1], ego[:, 3] = x, y, 3.0
    dev = BatchCoordinateConverter(path, len(x), engine=eng)
    host = BatchCoordinateConverter(path, len(x))
    dev.prev_s[:] = host.prev_s[:] = prev
    with np.errstate(all="ignore"):
        a, ok_a = ego_to_frenet_many(dev, np.arange(len(x)), ego, np.zeros(len(x)))
        b, ok_b = ego_to_frenet_many(host, np.arange(len(x)), ego, np.zeros(len(x)))
    assert np.array_equal(a, b, equal_nan=True) and np.array_equal(ok_a, ok_b)
    assert np.array_equal(dev.prev_s, host.prev_s, equal_nan=True)
    assert dev.host_rows == len(x) and dev.device_rows == 0


def _scatter(path, n, rng):
    """n egos scattered around the path and past both ends."""
    s = rng.uniform(-10.0, path.s[-1] + 10.0, n)
    px, py = path.calc_position(np.clip(s, 0.0, path.s[-1]))
    ego = np.zeros((n, 5))
    ego[:, 0] = px + np.minimum(s, 0.0) + np.maximum(s - path.s[-1], 0.0)
    ego[:, 1] = py + rng.normal(0.0, 1.5, n)
    ego[:, 2], ego[:, 3], ego[:, 4] = rng.normal(0.0, 0.2, n), rng.uniform(0.0, 9.0, n), rng.normal(0.0, 1.0, n)
    return ego


def test_large_batch_equals_the_host_converter():
    """10^5 rows, fresh caches then one step later with warm ones: the upload takes longer than the launch, so the
    kernel has to be ordered after it.  Checked through the engine and through the C entry point with a NULL stream
    behind an asynchronous upload on torch's default stream."""
    import ctypes as C
    import torch
    path = _curved_path()
    eng = _engine("curved")
    n = 100_000
    rng = np.random.default_rng(29)
    ego = _scatter(path, n, rng)
    kappa = rng.normal(0.0, 0.05, n)
    idx = np.arange(n)
    dev = BatchCoordinateConverter(path, n, engine=eng)
    host = BatchCoordinateConverter(path, n)
    for step in range(2):
        e = ego.copy()
        e[:, 0] += step * 0.4
        a, ok_a = ego_to_frenet_many(dev, idx, e, kappa)
        b, ok_b = ego_to_frenet_many(host, idx, e, kappa)
        assert np.array_equal(ok_a, ok_b) and np.array_equal(a, b, equal_nan=True), step
        assert np.array_equal(dev.prev_s, host.prev_s, equal_nan=True), step
    assert dev.device_rows >= 0.95 * 2 * n

    prev = np.where(rng.random(n) < 0.5, np.nan, host.prev_s)
    want_s, want_status = eng.nearest_s(ego[:, 0], ego[:, 1], prev)
    h_in = torch.from_numpy(np.concatenate([ego[:, 0], ego[:, 1], prev])).pin_memory()
    d_in = torch.empty_like(h_in, device=torch.device("cuda", eng.device))
    d_in.copy_(h_in, non_blocking=True)                              # legacy default stream, asynchronous
    s_out = torch.empty(n, dtype=torch.float64, device=d_in.device)
    st_out = torch.empty(n, dtype=torch.int32, device=d_in.device)
    p = d_in.data_ptr()
    rc = eng.lib.fot_nearest_s_device(eng._h, None, n, C.c_void_p(p), C.c_void_p(p + 8 * n), C.c_void_p(p + 16 * n),
                                      C.c_void_p(s_out.data_ptr()), C.c_void_p(st_out.data_ptr()))
    assert rc == 0
    assert np.array_equal(st_out.cpu().numpy(), want_status)
    assert np.array_equal(s_out.cpu().numpy(), want_s, equal_nan=True)


def test_recorded_reference_calls():
    """(c) Every recorded scenario_01 closed-loop call: ego, _prev_s and _last_kappa in, the reference's Frenet state
    out, bit for bit."""
    store = runners.load_golden("closed_loop_s01.npz")
    path = CubicSpline2D(list(store["waypoints_x"]), list(store["waypoints_y"]))
    n = len(store["kept"])
    cases = [runners.golden_case(store, f"c{j}") for j in range(n)]
    from integrated_path_planning_b200.batch import BatchFrenetPlanner
    pl = BatchFrenetPlanner(path, **scenarios.S1_KNOBS)
    dev = BatchCoordinateConverter(path, n, engine=pl.engine)
    dev.prev_s[:] = [float(g["prev_s"]) for g in cases]
    ego = np.stack([g["ego"] for g in cases])
    kappa = np.array([float(g["last_kappa"]) for g in cases])
    got, ok = ego_to_frenet_many(dev, np.arange(n), ego, kappa)
    assert ok.all()
    for j, g in enumerate(cases):
        assert np.array_equal(got[j], g["fs"]), (j, got[j] - g["fs"])
    assert dev.device_rows > 0


class _FailingRows(BatchCoordinateConverter):
    """Reports the conversion of converters `fail` as failed (the reference raises there and plan() returns None)."""

    def __init__(self, *a, fail=(), **kw):
        super().__init__(*a, **kw)
        self.fail = np.asarray(fail, dtype=np.int64)

    def reference_points(self, idx, x, y):
        out = super().reference_points(idx, x, y)
        out[-1][np.isin(idx, self.fail)] = False
        return out


def test_plan_batch_from_ego_equals_host_conversion_then_plan_batch():
    """(d) 512 config-4 egos: the same winners, costs, stats and winner series as the host conversion followed by
    plan_batch.  Rows whose conversion fails come back as plan()'s None."""
    import bench
    from integrated_path_planning_b200.batch import BatchFrenetPlanner
    n = 512
    spline = CubicSpline2D(*scenarios.STRAIGHT_60)
    pl = BatchFrenetPlanner(spline, **scenarios.S1_KNOBS)
    ego = np.empty((n, 5))
    dyn = np.empty((n, bench.N_PEDS, bench.T_OBS, 2))
    for i in range(n):
        e, d = bench.ego_and_field(i)
        ego[i], dyn[i] = e, d
    kappa = np.random.default_rng(5).normal(0.0, 0.02, n)

    host_conv = BatchCoordinateConverter(spline, n)
    fs, ok_host = ego_to_frenet_many(host_conv, np.arange(n), ego, kappa)
    ref = pl.plan_batch(fs, bench.TARGET_SPEED, dynamic_obstacles=dyn)
    want = {k: getattr(ref, k).copy() for k in ("best_idx", "best_cost", "stats", "winner_len", "winner")}

    got, ok = pl.plan_batch_from_ego(ego, bench.TARGET_SPEED, last_kappa=kappa, dynamic_obstacles=dyn)
    assert np.array_equal(ok, ok_host) and ok.all()
    assert np.array_equal(got.best_idx, want["best_idx"])
    assert np.array_equal(got.best_cost.view(np.int64), want["best_cost"].view(np.int64))
    assert np.array_equal(got.stats, want["stats"])
    assert np.array_equal(got.winner_len, want["winner_len"])
    for q in np.nonzero(want["best_idx"] >= 0)[0]:
        w = int(want["winner_len"][q])
        assert np.array_equal(got.winner[q, :, :w], want["winner"][q, :, :w]), q
    assert (want["best_idx"] >= 0).any() and (want["best_idx"] < 0).any()

    failed = np.arange(5, n, 41)
    conv = _FailingRows(spline, n, engine=pl.engine, fail=failed)
    got, ok = pl.plan_batch_from_ego(ego, bench.TARGET_SPEED, last_kappa=kappa, converter=conv, dynamic_obstacles=dyn)
    assert np.array_equal(np.nonzero(~ok)[0], failed)
    assert (got.best_idx[failed] == -1).all() and np.isinf(got.best_cost[failed]).all()
    assert (got.stats[failed] == 0).all() and (got.winner_len[failed] == 0).all()
    assert all(got.series(int(q)) is None for q in failed)
    assert np.array_equal(got.best_idx[ok], want["best_idx"][ok])
    assert np.array_equal(conv.prev_s, host_conv.prev_s, equal_nan=True)
    assert conv.device_rows > 0


def test_closed_loop_with_device_converters_equals_host_converters():
    """(e) 32 perturbed variants of rollout_s01: the whole run() with the device-backed converters equals the run
    with host converters."""
    from integrated_path_planning_b200.rollout import BatchedClosedLoop
    z = np.load(os.path.join(HERE, "golden", "rollout_s01.npz"))
    knobs = {k[5:]: float(z[k]) for k in z.files if k.startswith("knob/")}
    rng = np.random.default_rng(17)
    n_var = int(z["n_variants"])
    tracks, ego0 = [], []
    for i in range(32):
        v = i % n_var
        t = z[f"v{v}/traj"]
        tracks.append(t + rng.normal(0.0, 0.3, (1, t.shape[1], 2)))
        e = z[f"v{v}/ego0"].copy()
        e[1] += rng.normal(0.0, 0.3)
        e[3] = max(0.5, e[3] + rng.normal(0.0, 0.3))
        ego0.append(e)
    outs = []
    for on_device in (True, False):
        sim = BatchedClosedLoop(z["v0/wx"], z["v0/wy"], knobs, np.stack(tracks), np.stack(ego0))
        if not on_device:
            sim.plan_conv = BatchCoordinateConverter(sim.spline, sim.n)
            sim.goal_conv = BatchCoordinateConverter(sim.spline, sim.n)
        sim.warmup()
        outs.append(sim.run())
        if on_device:
            assert sim.plan_conv.device_rows > 0 and sim.goal_conv.device_rows > 0
    a, b = outs
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=a[k].dtype.kind == "f"), k


def test_certified_share_of_the_walks():
    """(f) The device answers at least 95 % of the rows of the random walks itself."""
    for name in sorted(PATHS):
        if name not in _SHARE:
            test_random_walks_equal_the_scalar_converter(name)
    dev = sum(d for d, _ in _SHARE.values())
    host = sum(h for _, h in _SHARE.values())
    assert dev / (dev + host) >= 0.95, _SHARE


_PROBE = r"""
#include "fot_frenet.cuh"
__global__ void cube_kernel(const double* dx, double* out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = fot::near_cube(dx[i]);
}
extern "C" int cube_probe(const double* dx, double* out, int n) {
  cube_kernel<<<(n + 255) / 256, 256>>>(dx, out, n);
  return (int)cudaDeviceSynchronize();
}
"""


def test_host_cube_within_the_assumed_ulps(tmp_path):
    """(g) The one assumption of the pinned positions: NumPy's `dx ** 3.0` lies within CUBE_ULPS ulps of the device's
    cube (fot::near_cube, compiled from the same header with the library's flags) for 10^6 offsets spread over the
    segments of the test paths."""
    import ctypes
    import torch
    from integrated_path_planning_b200 import build
    src = tmp_path / "cube_probe.cu"
    src.write_text(_PROBE)
    so = tmp_path / "cube_probe.so"
    cmd = [os.environ.get("NVCC", "nvcc"), *build.NVCC_FLAGS, "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(build.HERE, "csrc"), "-o", str(so), str(src)]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    assert proc.returncode == 0, proc.stdout + proc.stderr
    lib = ctypes.CDLL(str(so))
    lib.cube_probe.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
    rng = np.random.default_rng(23)
    dx = []
    for make in list(PATHS.values()) + [lambda: CubicSpline2D(*scenarios.STRAIGHT_60)]:
        knots = spline_tables(make())["knots"]
        seg = rng.integers(0, len(knots) - 1, 250_000)
        dx.append(rng.random(250_000) * (knots[seg + 1] - knots[seg]))
    dx = np.concatenate(dx)[:1_000_000]
    d_in = torch.from_numpy(dx).cuda()
    d_out = torch.empty_like(d_in)
    assert lib.cube_probe(d_in.data_ptr(), d_out.data_ptr(), len(dx)) == 0
    dev = d_out.cpu().numpy()
    assert (dx >= 0).all()
    # the host search cubes whole grids (global search), 100-sample rows (window) and 3-element arrays (refinement):
    # NumPy may take short arrays and loop tails through other code than its main SIMD loop, so each size is checked
    for chunk in (len(dx), 100, 3):
        host = np.concatenate([dx[k:k + chunk] ** 3.0 for k in range(0, len(dx), chunk)])
        ulps = np.abs(host.view(np.int64) - dev.view(np.int64))
        assert ulps.max() <= CUBE_ULPS, (chunk, int(ulps.max()))
