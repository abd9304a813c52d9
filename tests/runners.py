"""Run one tests.scenarios.Query through the oracle and through the CUDA planner, and compare."""
from __future__ import annotations

import numpy as np

from oracle import frenet_oracle as O
from tests.scenarios import Query

SERIES = ("t", "s", "s_d", "s_dd", "s_ddd", "d", "d_d", "d_dd", "d_ddd", "x", "y", "yaw", "c", "v", "a")
RTOL = 1e-9      # north_star: "trajectory points and costs must agree within 1e-9 relative in fp64"
ATOL = 1e-9      # for samples that are mathematically zero (jerk on a straight, yaw on y=0, ...)


class _Ego:
    def __init__(self, x, y, yaw, v, a):
        self.x, self.y, self.yaw, self.v, self.a = x, y, yaw, v, a


def reload_options():
    """The FOT_* tuning variables are resolved when a handle is created; tests that switch variants on a live
    planner change the environment and then ask every live handle to re-read it (fot_reload_options(NULL))."""
    from integrated_path_planning_b200 import _lib
    _lib.check(_lib.load().fot_reload_options(None), "fot_reload_options")


class fot_env:
    """with fot_env(FOT_SWEEP="items"): ...   -- environment change + option reload, restored on exit."""

    def __init__(self, **kv):
        self.kv = kv

    def __enter__(self):
        import os
        self.old = {k: os.environ.get(k) for k in self.kv}
        os.environ.update({k: str(v) for k, v in self.kv.items()})
        reload_options()

    def __exit__(self, *a):
        import os
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        reload_options()


def make_footprint(spec):
    """EgoFootprint.multi_circle restated (reference src/core/footprint.py:66-81)."""
    if spec is None:
        return None
    length, width, n = spec
    seg = length / n
    offsets = -length / 2 + seg / 2 + seg * np.arange(n)
    radius = float(np.hypot(seg / 2, width / 2))

    class FP:
        pass
    fp = FP()
    fp.offsets, fp.radius = offsets, radius
    return fp


def oracle_planner(q: Query) -> O.OraclePlanner:
    kn = O.Knobs(**q.knobs)
    fp = make_footprint(q.footprint)
    if fp is not None:
        kn.footprint_offsets, kn.footprint_radius = fp.offsets, fp.radius
    pl = O.OraclePlanner(O.Spline2D(*q.waypoints), kn)
    pl.last_kappa = q.last_kappa
    return pl


def run_oracle(q: Query) -> O.OracleResult:
    static = np.empty((0, 2)) if q.static is None else q.static
    return oracle_planner(q).plan(q.ego, static, q.dyn, q.target_speed, q.overrides, q.dist, q.max_stop_distance)


def cuda_planner(q: Query, device=0):
    from integrated_path_planning_b200 import CubicSpline2D, FrenetPlanner
    pl = FrenetPlanner(CubicSpline2D(*q.waypoints), footprint=make_footprint(q.footprint), device=device, **q.knobs)
    pl._last_kappa = q.last_kappa
    return pl


def run_cuda(q: Query, planner=None):
    pl = planner or cuda_planner(q)
    static = np.empty((0, 2)) if q.static is None else q.static
    path = pl.plan(_Ego(*q.ego), static, q.dyn, q.target_speed, q.overrides, q.dist, q.max_stop_distance,
                   _want_candidates=True)
    return pl, path


def assert_matches_oracle(q: Query, ref: O.OracleResult, pl, path, exact_counts=True):
    """The parity bar: identical winner index, categories and stats; values within 1e-9."""
    res = pl.last_result
    n_c = len(ref.categories)
    assert int(res.n_cand[0]) == n_c, (q.name, int(res.n_cand[0]), n_c)
    cats = res.cand_cat[0, :n_c].astype(np.int8)
    mism = np.nonzero(cats != ref.categories)[0]
    assert mism.size == 0, (q.name, "category mismatch", mism[:10], cats[mism[:10]], ref.categories[mism[:10]])
    np.testing.assert_allclose(res.cand_cost[0, :n_c], ref.costs, rtol=RTOL, atol=0, err_msg=q.name + " costs")
    assert pl.last_check_stats == ref.stats, (q.name, pl.last_check_stats, ref.stats)
    assert int(res.best_idx[0]) == ref.best_index, (q.name, int(res.best_idx[0]), ref.best_index)
    if ref.best_index < 0:
        assert path is None
        return
    assert path is not None
    np.testing.assert_allclose(float(path.cost), ref.cost, rtol=RTOL, atol=0)
    for name in SERIES:
        got = np.asarray(getattr(path, name), dtype=float)
        want = ref.arrays[name]
        assert got.shape == want.shape, (q.name, name, got.shape, want.shape)
        np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL, err_msg=f"{q.name} {name}")


def bit_exact_report(ref: O.OracleResult, pl, path) -> dict:
    """How much of the output is bit-identical (informational; the bar is 1e-9)."""
    res = pl.last_result
    n_c = len(ref.categories)
    out = {"cost_bit_exact_frac": float(np.mean(res.cand_cost[0, :n_c] == ref.costs))}
    if path is not None and ref.arrays is not None:
        for name in SERIES:
            out[name] = float(np.mean(np.asarray(getattr(path, name), dtype=float) == ref.arrays[name]))
    return out


# ---------------------------------------------------------------------------------------------
# golden fixtures (made by tests/golden/make_golden.py from the unmodified reference)
# ---------------------------------------------------------------------------------------------
import os as _os

GOLDEN_DIR = _os.path.join(_os.path.dirname(_os.path.abspath(__file__)), "golden")
GOLDEN_STAT_KEYS = ("ok", "max_speed_error", "max_accel_error", "max_curvature_error", "max_lat_accel_error",
                    "road_bound_error", "collision_error", "stop_distance_error")


def load_golden(name):
    return np.load(_os.path.join(GOLDEN_DIR, name))


def golden_case(store, prefix):
    """One recorded reference plan() result as a dict."""
    out = {k[len(prefix) + 1:]: store[k] for k in store.files if k.startswith(prefix + "/")}
    out["stats_dict"] = {k: int(v) for k, v in zip(GOLDEN_STAT_KEYS, out["stats"]) if v >= 0}
    return out


def assert_oracle_matches_golden(name, res: O.OracleResult, g, rtol=1e-12):
    """Oracle vs the recorded reference: identical decisions; values to 1e-12 (bit-identical on the
    machine that made the fixtures; a different host libm/BLAS may move the last bits)."""
    assert np.array_equal(res.categories.astype(np.uint8), g["cats"]), name
    np.testing.assert_allclose(res.costs, g["costs"], rtol=rtol, atol=0, err_msg=name)
    assert res.best_index == int(g["best"]), (name, res.best_index, int(g["best"]))
    assert res.stats == g["stats_dict"], (name, res.stats, g["stats_dict"])
    np.testing.assert_allclose(np.array(res.frenet_state), g["fs"], rtol=rtol, atol=1e-15, err_msg=name)
    if res.best_index >= 0:
        np.testing.assert_allclose(res.cost, float(g["cost"]), rtol=rtol)
        for s in SERIES:
            if "w_" + s in g:
                np.testing.assert_allclose(res.arrays[s], g["w_" + s], rtol=1e-10, atol=1e-10, err_msg=f"{name} {s}")


def assert_cuda_matches_golden(name, pl, path, g):
    """CUDA planner vs the recorded reference: the north-star bar (index identical, 1e-9 on values)."""
    res = pl.last_result
    n_c = len(g["cats"])
    assert int(res.n_cand[0]) == n_c, (name, int(res.n_cand[0]), n_c)
    cats = res.cand_cat[0, :n_c]
    mism = np.nonzero(cats != g["cats"])[0]
    assert mism.size == 0, (name, "category mismatch", mism[:10], cats[mism[:10]], g["cats"][mism[:10]])
    np.testing.assert_allclose(res.cand_cost[0, :n_c], g["costs"], rtol=RTOL, atol=0, err_msg=name)
    assert pl.last_check_stats == g["stats_dict"], (name, pl.last_check_stats, g["stats_dict"])
    assert int(res.best_idx[0]) == int(g["best"]), (name, int(res.best_idx[0]), int(g["best"]))
    if int(g["best"]) < 0:
        assert path is None
        return
    np.testing.assert_allclose(float(path.cost), float(g["cost"]), rtol=RTOL)
    for s in SERIES:
        if "w_" + s in g:
            got = np.asarray(getattr(path, s), dtype=float)
            assert got.shape == g["w_" + s].shape, (name, s)
            np.testing.assert_allclose(got, g["w_" + s], rtol=RTOL, atol=ATOL, err_msg=f"{name} {s}")
