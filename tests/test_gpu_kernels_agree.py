"""GPU: the two sweep kernels are independent implementations of the same contract -- the
pair-per-warp `fot_sweep_pairs` (default) and the sample-major `fot_sweep_items` (FOT_SWEEP=items, also
the kernel for shapes beyond the pair kernel's limits).  They must agree bit for bit on every
candidate's category and cost, on the winner and on the histogram, at sizes the NumPy oracle cannot reach."""
import os

import numpy as np
import pytest

from tests import scenarios

pytestmark = pytest.mark.gpu


def _run(kernel, fn):
    from tests import runners
    with runners.fot_env(FOT_SWEEP=kernel):      # options are resolved per handle: reload after the switch
        return fn()


def _assert_same(a, b):
    assert np.array_equal(a.n_cand, b.n_cand)
    assert np.array_equal(a.cand_cat, b.cand_cat)
    n = int(a.n_cand.max())
    assert np.array_equal(a.cand_cost[:, :n].view(np.uint64), b.cand_cost[:, :n].view(np.uint64))
    assert np.array_equal(a.best_idx, b.best_idx)
    assert np.array_equal(a.best_cost.view(np.uint64), b.best_cost.view(np.uint64))
    assert np.array_equal(a.stats, b.stats)
    assert np.array_equal(a.winner_len, b.winner_len)


def _planner(knobs, wp):
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    return BatchFrenetPlanner(CubicSpline2D(*wp), **knobs)


def test_config4_batch_both_kernels():
    """512 queries of BASELINE config 4 (1261 candidates x 50 pedestrians each)."""
    import bench
    _, frenet, dyn = bench.make_queries(1000, 512)
    pl = _planner(scenarios.S1_KNOBS, scenarios.STRAIGHT_60)
    run = lambda: pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0], want_candidates=True)
    b, d = _run("items", run), _run("pairs", run)
    _assert_same(b, d)
    assert (b.stats[:, 6] > 0).any() and (b.best_idx >= 0).any()


def test_curved_path_state_machine_knobs_both_kernels():
    """S-curve reference line, per-query target speeds / limits / stop distances (the state machine's
    three knob sets), static wall and dynamic field together."""
    rng = np.random.default_rng(3)
    n = 96
    wp = scenarios.s_curve_waypoints()
    frenet = np.stack([rng.uniform(2, 30, n), rng.uniform(0, 8, n), rng.uniform(-1, 1, n),
                       rng.uniform(-1.5, 1.5, n), rng.normal(0, 0.3, n), rng.normal(0, 0.05, n)], axis=1)
    k = scenarios.S1_KNOBS
    target = np.tile([6.0, 3.6, 0.0], n // 3)
    limits = np.tile([[k["max_speed"], k["max_accel"], k["max_curvature"], k["max_lat_accel"]],
                      [k["max_speed"] * 0.6, k["max_accel"] * 1.5, k["max_curvature"], k["max_lat_accel"]],
                      [k["max_speed"], k["max_accel"] * 3.0, k["max_curvature"], k["max_lat_accel"] * 2.0]], (n // 3, 1))
    msd = np.where(target == 0.0, 5.0, np.nan)
    dyn = np.stack([scenarios.pedestrian_field(np.random.default_rng(50 + i), 30, x_range=(0.0, 70.0), y_range=(-8.0, 8.0))
                    for i in range(n)])
    wall = scenarios.wall(x=45.0, half=1.0, n=9)
    pl = _planner(k, wp)
    run = lambda: pl.plan_batch(frenet, target, dynamic_obstacles=dyn, static_obstacles=wall, limits=limits,
                                max_stop_distance=msd, want_candidates=True)
    b, d = _run("items", run), _run("pairs", run)
    _assert_same(b, d)


def test_dense_grid_distribution_both_kernels():
    """BASELINE config 3: 65 d x 32 T x 32 v (+ brake ladder) = 66.5k candidates against 200 pedestrians
    x 20 samples (chance-constrained, epsilon = 0) -- 9.4e9 dense evaluations in one plan() call."""
    rng = np.random.default_rng(33)
    knobs = dict(scenarios.S1_KNOBS, d_road_w=0.1, max_road_width=3.2, min_t=1.9, max_t=5.0, d_t_s=0.2)
    wp = (np.linspace(0.0, 80.0, 9).tolist(), [0.0] * 9)
    base = scenarios.pedestrian_field(rng, 200, x_range=(5.0, 65.0), vel_clip=2.5)
    dist = scenarios.sample_distribution(rng, base, 20)
    pl = _planner(knobs, wp)
    fs = np.array([[5.0, 5.0, 0.0, 0.0, 0.0, 0.0]])
    run = lambda: pl.plan_batch(fs, 6.2, distribution=dist[None], want_candidates=True)
    a, d = _run("items", run), _run("pairs", run)
    _assert_same(a, d)
    assert int(a.n_cand[0]) > 60000


def test_budgeted_distribution_and_footprint_both_kernels():
    """chance_epsilon > 0 (violation budget per candidate) and a 3-circle footprint on an arc."""
    rng = np.random.default_rng(5)
    n = 24
    knobs = dict(scenarios.S1_KNOBS, chance_epsilon=0.25)
    wp = scenarios.arc_waypoints()
    frenet = np.stack([rng.uniform(1, 10, n), rng.uniform(1, 7, n), rng.uniform(-1, 1, n),
                       rng.uniform(-1, 1, n), rng.normal(0, 0.2, n), rng.normal(0, 0.05, n)], axis=1)
    dists = []
    for i in range(n):
        r = np.random.default_rng(200 + i)
        base = scenarios.pedestrian_field(r, 14, x_range=(0.0, 20.0), y_range=(-5.0, 25.0))
        dists.append(scenarios.sample_distribution(r, base, 12, sigma=0.08))
    dist = np.stack(dists)
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    from tests import runners
    pl = BatchFrenetPlanner(CubicSpline2D(*wp), footprint=runners.make_footprint((4.5, 2.0, 3)), **knobs)
    run = lambda: pl.plan_batch(frenet, 6.0, distribution=dist, want_candidates=True)
    b, d = _run("items", run), _run("pairs", run)
    _assert_same(b, d)


def test_campaign_shape_instantiations_of_the_pair_kernel():
    """fot_sweep_pairs compiles the planning-campaign shape (no static obstacles, one circle, no violation budget, no
    per-candidate outputs) into instantiations of its own, resident and gated.  Winners, costs, histograms and the
    returned series must be those of the general instantiation and of fot_sweep_items, bit for bit."""
    import torch
    import bench
    from integrated_path_planning_b200 import _lib
    from integrated_path_planning_b200.batch import DeviceBatch
    from tests import runners
    _, frenet, dyn = bench.make_queries(2000, 384)
    pl = _planner(scenarios.S1_KNOBS, scenarios.STRAIGHT_60)
    keys = ("best_idx", "best_cost", "stats", "winner_len", "winner")

    def resident():
        db = DeviceBatch(pl, frenet, 6.0, dyn, _lib.FOT_DYN_SINGLE)
        db.launch()
        torch.cuda.synchronize()
        kind = int(pl.engine.lib.fot_last_sweep_kind(pl.engine._h))
        return {k: db.out[k].cpu().numpy().copy() for k in keys}, kind

    def host():
        r = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0])
        return {k: np.array(getattr(r, k)) for k in keys}

    def same(a, b):
        for k in ("best_idx", "stats", "winner_len"):
            assert np.array_equal(a[k], b[k]), k
        assert np.array_equal(a["best_cost"].view(np.uint64), b["best_cost"].view(np.uint64))
        n_t = a["winner"].shape[-1]
        live = (np.arange(n_t)[None, None, :] < a["winner_len"].reshape(-1, 1, 1)) & (a["best_idx"].reshape(-1, 1, 1) >= 0)
        wa, wb = a["winner"].reshape(len(a["best_idx"]), -1, n_t), b["winner"].reshape(len(b["best_idx"]), -1, n_t)
        assert np.array_equal(np.where(live, wa, 0.0).view(np.uint64), np.where(live, wb, 0.0).view(np.uint64))

    pl.engine
    with runners.fot_env(FOT_SWEEP="items"):
        ref, kind = resident()
        assert kind == 1
        ref_host = host()
    same(ref, ref_host)
    for env in (dict(), dict(FOT_PAIR_SIMPLE=0)):
        with runners.fot_env(**env):
            got, kind = resident()
            assert kind == 4
            same(ref, got)
            same(ref, host())
    assert (ref["best_idx"] >= 0).sum() > 100


def test_random_shapes_pair_kernel_against_item_kernel():
    """Shape fuzz for the pair kernel's compile-time layout, clamped quads and tail masks: time grids from 8 to 56
    samples (one pass, exactly 32 / 33 samples, two passes), 1 to 95 lateral targets (quads with 1-3 live candidates), one
    to many terminal speeds, brake ladder on and off, obstacle horizons shorter and longer than the time grid, static
    obstacles across chunk borders, single-sample and distribution mode with and without a violation budget, with and
    without a footprint -- every candidate's category and cost, winners and histograms bit for bit against
    fot_sweep_items, and the winners once more through the instantiation without per-candidate outputs."""
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    from tests import runners
    rng = np.random.default_rng(77)
    paths = (scenarios.STRAIGHT_60, scenarios.s_curve_waypoints(), scenarios.arc_waypoints())
    seen_kinds, seen_feats = set(), set()
    for case in range(28):
        dt = float(rng.choice([0.1, 0.2, 0.25]))
        n_max = int(rng.choice([8, 17, 31, 32, 33, 40, 47, 56]))
        max_t = round((n_max - 1) * dt, 6)
        min_t = round(max(dt * 4, max_t - dt * int(rng.integers(0, 6))), 6)
        n_side = int(rng.choice([0, 1, 2, 5, 9, 16, 31, 47]))
        road = 2.7
        knobs = dict(scenarios.S1_KNOBS, dt=dt, min_t=min_t, max_t=max_t, max_road_width=road,
                     d_road_w=(road / (n_side + 0.5) if n_side > 0 else 2 * road + 1.0),
                     d_t_s=float(rng.choice([0.5, 5.0 / 3.6, 3.0, 20.0])))
        if case % 4 == 3:
            knobs["chance_epsilon"] = float(rng.choice([0.0, 0.2, 0.34]))
        footprint = runners.make_footprint((4.5, 2.0, 3)) if case % 5 == 4 else None
        pl = BatchFrenetPlanner(CubicSpline2D(*paths[case % 3]), footprint=footprint, **knobs)
        n = 12
        frenet = np.stack([rng.uniform(2, 20, n), rng.uniform(0, 8, n), rng.uniform(-1, 1, n), rng.uniform(-1.5, 1.5, n),
                           rng.normal(0, 0.3, n), rng.normal(0, 0.05, n)], axis=1)
        frenet[::5, 1] = rng.uniform(0.0, 0.1, len(frenet[::5]))                   # too slow for the brake ladder
        target = rng.choice([0.0, 2.0, 6.0, 8.5], n)
        t_obs = int(rng.choice([1, 5, n_max - 3, n_max, n_max + 9]))
        t_obs = max(1, t_obs)
        n_ped = int(rng.choice([1, 7, 31, 33, 70]))
        kw = {}
        if case % 4 == 3:
            S = int(rng.choice([3, 6]))
            base = np.stack([scenarios.pedestrian_field(rng, min(n_ped, 12), n_steps=t_obs, dt=dt, x_range=(0.0, 40.0), y_range=(-6.0, 6.0)) for _ in range(n)])
            kw["distribution"] = np.stack([scenarios.sample_distribution(rng, base[i], S, sigma=0.08) for i in range(n)])
        else:
            kw["dynamic_obstacles"] = np.stack([scenarios.pedestrian_field(rng, n_ped, n_steps=t_obs, dt=dt, x_range=(0.0, 40.0), y_range=(-6.0, 6.0))
                                                for _ in range(n)])
        if case % 3 == 1:
            m = int(rng.choice([1, 30, 40, 75]))
            kw["static_obstacles"] = np.stack([rng.uniform(5.0, 45.0, m), rng.uniform(-5.0, 5.0, m)], axis=1)
        msd = np.where(target == 0.0, 6.0, np.nan)
        run = lambda cands: pl.plan_batch(frenet, target, max_stop_distance=msd, want_candidates=cands, **kw)
        pl.engine
        with runners.fot_env(FOT_SWEEP="items"):
            ref = run(True)
        got = run(True)
        seen_kinds.add(int(pl.engine.lib.fot_last_sweep_kind(pl.engine._h)))
        seen_feats.add(int(pl.engine.lib.fot_last_pair_features(pl.engine._h)))
        _assert_same(ref, got)
        lean = run(False)
        seen_feats.add(int(pl.engine.lib.fot_last_pair_features(pl.engine._h)))
        assert np.array_equal(ref.best_idx, lean.best_idx) and np.array_equal(ref.stats, lean.stats), case
        assert np.array_equal(ref.best_cost.view(np.uint64), lean.best_cost.view(np.uint64)), case
        if case % 2 == 0:
            with runners.fot_env(FOT_PAIR_SIMPLE=0):                               # the instantiation with every mode compiled in
                _assert_same(ref, run(True))
                assert int(pl.engine.lib.fot_last_pair_features(pl.engine._h)) in (31, -1)
    assert 4 in seen_kinds
    # the kernel is compiled per mode set (campaign shape, + statics, + outputs, + both, budget, statics + footprint,
    # everything; the unstaged set runs in the config-3 tests): these ran here
    assert {0, 1, 8, 9, 31} <= seen_feats, seen_feats
