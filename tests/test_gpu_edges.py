"""GPU: edge cases of the sample-major sweep that the seeded queries do not reach -- non-finite states,
negative limits, the full-queue path of the collision phase, obstacle horizons longer than the time grid,
unstaged obstacle fields, one block per CTA vs one query per CTA."""
import os

import numpy as np
import pytest

from oracle import frenet_oracle as O
from tests import runners, scenarios

pytestmark = pytest.mark.gpu


def _planner(knobs=None, wp=scenarios.STRAIGHT_60):
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    return BatchFrenetPlanner(CubicSpline2D(*wp), **(knobs or scenarios.S1_KNOBS))


def _oracle(knobs=None, wp=scenarios.STRAIGHT_60):
    return O.OraclePlanner(O.Spline2D(*wp), O.Knobs(**(knobs or scenarios.S1_KNOBS)))


def _env(**kv):
    class _Ctx:
        def __enter__(self):
            self.old = {k: os.environ.get(k) for k in kv}
            os.environ.update({k: str(v) for k, v in kv.items()})
            runners.reload_options()

        def __exit__(self, *a):
            for k, v in self.old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
            runners.reload_options()
    return _Ctx()


def _same(name, v, w, lens=None):
    """Bit-for-bit equality of two result arrays; winner rows only up to winner_len (the padding is never written)."""
    if name == "winner" and lens is not None:
        keep = np.arange(v.shape[-1])[None, None, :] < np.asarray(lens)[:, None, None]
        v, w = np.where(keep, v, 0.0), np.where(keep, w, 0.0)
    return np.array_equal(v.view(np.uint64), w.view(np.uint64)) if v.dtype == np.float64 else np.array_equal(v, w)


def _check(res, refs):
    for i, ref in enumerate(refs):
        n_c = len(ref.categories)
        assert int(res.n_cand[i]) == n_c
        assert np.array_equal(res.cand_cat[i, :n_c].astype(np.int8), ref.categories), i
        assert int(res.best_idx[i]) == ref.best_index
        assert res.stats[i].tolist() == [ref.stats.get(k, 0) for k in runners.GOLDEN_STAT_KEYS]


def test_non_finite_states_drop_every_candidate():
    """NaN / inf anywhere in the Frenet state: the reference's empty / non-finite guards drop all candidates
    silently (histogram all zero, no path); finite neighbours in the same batch are unaffected."""
    dyn = scenarios.pedestrian_field(np.random.default_rng(1), 5)
    states = np.array([[5.0, np.nan, 0, 0, 0, 0], [5.0, 5.0, 0.0, np.inf, 0.0, 0.0], [np.nan, 5, 0, 0, 0, 0],
                       [5.0, 5.0, 0.0, 0.1, 0.0, 0.0]])
    pl, orc = _planner(), _oracle()
    res = pl.plan_batch(states, 6.0, dynamic_obstacles=np.stack([dyn] * 4), want_candidates=True)
    refs = [orc.plan_frenet(tuple(s), np.empty((0, 2)), dyn, 6.0) for s in states]
    _check(res, refs)
    assert res.best_idx[:3].tolist() == [-1, -1, -1] and res.stats[:3].sum() == 0 and res.best_idx[3] >= 0


def test_negative_limits_reject_everything():
    """`abs(a) > negative` is true for every checked sample: the squared device tests must agree."""
    dyn = scenarios.pedestrian_field(np.random.default_rng(2), 4)
    fs = np.array([[5.0, 5.0, 0.0, 0.0, 0.0, 0.0]])
    pl, orc = _planner(), _oracle()
    for key, col in (("max_accel", 1), ("max_speed", 0), ("max_curvature", 2), ("max_lat_accel", 3)):
        lim = pl.resolve_limits({key: -1.0})
        res = pl.plan_batch(fs, 6.0, dynamic_obstacles=dyn[None], limits=lim, want_candidates=True)
        _check(res, [orc.plan_frenet(tuple(fs[0]), np.empty((0, 2)), dyn, 6.0, {key: -1.0})])
        assert res.best_idx[0] == -1


def test_full_collision_queue_degrades_to_in_place_tests():
    """A dense crowd in the lane with the queue capped at 4 entries: every survivor of the window test is
    tested by the thread that found it; results must not change."""
    rng = np.random.default_rng(3)
    n = 12
    frenet = np.stack([rng.uniform(2, 15, n), rng.uniform(1, 7, n), rng.uniform(-1, 1, n), rng.uniform(-1, 1, n),
                       rng.normal(0, 0.2, n), rng.normal(0, 0.05, n)], axis=1)
    dyn = np.stack([scenarios.pedestrian_field(np.random.default_rng(40 + i), 60, y_range=(-3.5, 3.5)) for i in range(n)])
    wall = scenarios.wall(x=33.0, half=1.5, n=13)
    pl = _planner()
    run = lambda: pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn, static_obstacles=wall, want_candidates=True)
    base = run()
    with _env(FOT_SWEEP="items"):                          # the sample-major kernel (the default is fot_sweep_pairs)
        items = run()
    with _env(FOT_SWEEP="items", FOT_QCAP=4):
        capped = run()
    with _env(FOT_SWEEP="items", FOT_STAGE_DYN=0, FOT_BPC=1):
        unstaged = run()
    with _env(FOT_STAGE_DYN=0, FOT_PAIR_CPQ=8):
        unstaged_pairs = run()
    for other in (items, capped, unstaged, unstaged_pairs):
        assert np.array_equal(base.cand_cat, other.cand_cat)
        assert np.array_equal(base.best_idx, other.best_idx) and np.array_equal(base.stats, other.stats)
        assert np.array_equal(base.best_cost.view(np.uint64), other.best_cost.view(np.uint64))
    orc = _oracle()
    _check(base, [orc.plan_frenet(tuple(frenet[i]), wall, dyn[i], 6.0) for i in range(3)])
    assert base.stats[:, 6].sum() > 0


def test_obstacle_horizon_longer_than_the_time_grid_and_single_step():
    """T_obs = 80 > 51 samples (extra steps are never indexed) and T_obs = 1 (every sample clamps to it)."""
    fs = np.array([[5.0, 5.0, 0.0, 0.2, 0.0, 0.0]])
    pl, orc = _planner(), _oracle()
    long = scenarios.pedestrian_field(np.random.default_rng(5), 9, n_steps=80)
    long[:, 60:] = [12.0, 0.0]                                # would block the lane if those steps were used
    res = pl.plan_batch(fs, 6.0, dynamic_obstacles=long[None], want_candidates=True)
    _check(res, [orc.plan_frenet(tuple(fs[0]), np.empty((0, 2)), long, 6.0)])
    one = scenarios.pedestrian_field(np.random.default_rng(6), 9, n_steps=1)
    res = pl.plan_batch(fs, 6.0, dynamic_obstacles=one[None], want_candidates=True)
    _check(res, [orc.plan_frenet(tuple(fs[0]), np.empty((0, 2)), one, 6.0)])


def test_many_speeds_split_a_horizon_over_several_blocks():
    """n_v = 16 terminal speeds do not fit one block of 320 threads (6 pairs x 51 samples): the horizon is cut
    into chunks of pairs; d_t_s small, coarse lateral grid to keep the oracle fast."""
    knobs = dict(scenarios.S1_KNOBS, d_t_s=0.4, d_road_w=0.9, min_t=4.6, max_t=5.0)
    fs = np.array([[5.0, 5.0, 0.0, 0.2, 0.0, 0.0], [8.0, 2.0, 0.5, -0.4, 0.1, 0.0]])
    dyn = np.stack([scenarios.pedestrian_field(np.random.default_rng(70 + i), 20) for i in range(2)])
    pl, orc = _planner(knobs), _oracle(knobs)
    res = pl.plan_batch(fs, 6.0, dynamic_obstacles=dyn, want_candidates=True)
    _check(res, [orc.plan_frenet(tuple(fs[i]), np.empty((0, 2)), dyn[i], 6.0) for i in range(2)])
    assert int(res.n_cand[0]) == 5 * 16 * 7 + 9            # 5 horizons x 16 speeds x 7 offsets + 9 brake horizons below min_t = 4.6


def test_host_chunking_and_cta_grouping_do_not_change_results():
    """1500 queries (not a multiple of the wave size): the pipelined, chunked host path with one CTA per query
    against a single launch with one block per CTA."""
    import bench
    _, frenet, dyn = bench.make_queries(5000, 250)
    frenet, dyn = np.tile(frenet, (6, 1)), np.tile(dyn, (6, 1, 1, 1, 1))
    pl = _planner()
    a = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0], want_candidates=True)
    a = {k: getattr(a, k).copy() for k in ("best_idx", "best_cost", "stats", "cand_cat", "winner", "winner_len")}
    with _env(FOT_HOST_CHUNKS=1, FOT_BPC=1):
        b = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0], want_candidates=True)
    for k, v in a.items():
        assert _same(k, v, getattr(b, k), a["winner_len"]), k
    assert np.array_equal(a["best_idx"][:250], a["best_idx"][250:500])


def test_gated_upload_pipeline_matches_the_single_launch():
    """The host-pointer call launches the sweep while the obstacle tensor is still being uploaded: CTAs wait for
    the slice of their query and box the predicted trajectories themselves.  Every variant of that pipeline
    (gated, chunked on two streams, odd slice and range counts, flags by copy instead of stream write)
    has to return what one plain launch over the resident tensor returns -- including queries with a NaN
    trajectory, whose box is NaN (fp.py:1211-1222), and a shared static wall."""
    import bench
    _, frenet, dyn = bench.make_queries(7000, 200)
    frenet, dyn = np.tile(frenet, (6, 1)), np.tile(dyn, (6, 1, 1, 1, 1)).copy()
    dyn[3::17, 0, 5, 20:, :] = np.nan                      # a pedestrian whose prediction breaks off
    dyn[8::29, 0, 2, 0, 1] = np.nan
    wall = np.stack([np.full(12, 30.0), np.linspace(-3.0, 3.0, 12)], axis=1)
    pl = _planner()
    keys = ("best_idx", "best_cost", "stats", "cand_cat", "winner", "winner_len")
    run = lambda: pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0], static_obstacles=wall, want_candidates=True)
    with _env(FOT_HOST_CHUNKS=1):
        ref = run()
        ref = {k: getattr(ref, k).copy() for k in keys}
    assert len(set(ref["best_idx"].tolist())) > 20
    variants = [dict(), dict(FOT_SWEEP="items"), dict(FOT_SWEEP="items", FOT_GATED=0), dict(FOT_GATED=0), dict(FOT_GATE_UPLOADS=7),
                dict(FOT_GATE_UPLOADS=64), dict(FOT_GATE_MEMCPY=1, FOT_HOST_CHUNKS=5),
                dict(FOT_STAGE_DYN=0), dict(FOT_GATED=0, FOT_HOST_CHUNKS=1, FOT_FUSED_BOX=1),
                dict(FOT_SWEEP="items", FOT_GATED=0, FOT_HOST_CHUNKS=1, FOT_FUSED_BOX=1)]
    for env in variants:
        with _env(**env):
            got = run()
        for k, v in ref.items():
            assert _same(k, v, getattr(got, k), ref["winner_len"]), (env, k)


def test_validity_screens_agree_with_the_oracle_near_the_limits():
    """Phase C settles several tests once per item for the whole grid of lateral targets (ends of the grid for the
    affine / convex ones, interval bounds for the rest) and skips the candidate loop for warps of clean items.
    Limits drawn right through the range the candidates actually take -- speeds, accelerations, curvatures,
    lateral accelerations and road widths that cut the grid -- put many items on the boundary of every screen; the
    categories of all candidates must still be the reference's, on a straight and on a curved path."""
    rng = np.random.default_rng(11)
    cases = []
    for k in range(14):
        over = dict(max_speed=float(rng.uniform(2.0, 9.0)), max_accel=float(rng.uniform(0.3, 3.0)),
                    max_curvature=float(rng.uniform(0.01, 0.3)), max_lat_accel=float(rng.uniform(0.05, 2.0)))
        fs = np.array([rng.uniform(3, 25), rng.uniform(0.0, 9.0), rng.uniform(-1.5, 1.5), rng.uniform(-2.9, 2.9),
                       rng.uniform(-1.0, 1.0), rng.uniform(-0.5, 0.5)])
        cases.append((over, fs, float(rng.uniform(0.5, 9.0))))
    for wp in (scenarios.STRAIGHT_60, scenarios.s_curve_waypoints(), scenarios.arc_waypoints()):
        for road in (2.7, 1.1):
            knobs = dict(scenarios.S1_KNOBS, max_road_width=road)
            pl, orc = _planner(knobs, wp), _oracle(knobs, wp)
            for over, fs, target in cases:
                dyn = scenarios.pedestrian_field(rng, 6)
                res = pl.plan_batch(fs[None], target, dynamic_obstacles=dyn[None], limits=pl.resolve_limits(over),
                                    want_candidates=True)
                _check(res, [orc.plan_frenet(tuple(fs), np.empty((0, 2)), dyn, target, over)])


def test_device_inputs_host_results_entry_point_matches_the_resident_launch():
    """fot_plan_batch_device_to_host: device-resident batch, winners delivered to host arrays range by range.
    Same bits as the plain launch followed by a read-back, for a batch that is cut into three ranges and for a
    small one that is not."""
    import torch
    import bench
    from integrated_path_planning_b200 import DeviceBatch, _lib
    pl = _planner()
    for count, tile in ((230, 6), (40, 1)):
        _, frenet, dyn = bench.make_queries(9000, count)
        frenet, dyn = np.tile(frenet, (tile, 1)), np.tile(dyn, (tile, 1, 1, 1, 1))
        batch = DeviceBatch(pl, frenet, 6.0, dyn, _lib.FOT_DYN_SINGLE)
        batch.launch(None)
        want = {k: v.cpu() for k, v in batch.out.items()}
        host = {k: torch.full(v.shape, -7, dtype=v.dtype).pin_memory() for k, v in batch.out.items()}
        batch.launch_to_host(host, torch.cuda.current_stream().cuda_stream)
        for k in want:
            a, b = want[k].numpy(), host[k].numpy()
            if k == "winner":                                  # rows are defined up to winner_len; the padding is not written
                n = want["winner_len"].numpy()
                for q in range(a.shape[0]):
                    assert np.array_equal(a[q, :, :n[q]].view(np.uint64), b[q, :, :n[q]].view(np.uint64)), (count * tile, q)
                continue
            same = np.array_equal(a.view(np.uint64), b.view(np.uint64)) if a.dtype == np.float64 else np.array_equal(a, b)
            assert same, (count * tile, k)


def test_compact_winner_read_back_and_fetch():
    """fot_result_t.winner_samples = k: the host-result calls copy back only the first k samples of every winner series
    (a closed-loop caller consumes sample 1, integrated_simulator.py:660-667); fot_fetch_winners reads full series of the
    last call from the device.  Both must be the bits of the full read-back, for a gated batch, a chunked one and a
    single plan()-sized call."""
    import bench
    for count, tile in ((230, 6), (3, 1)):
        _, frenet, dyn = bench.make_queries(11000, count)
        frenet, dyn = np.tile(frenet, (tile, 1)), np.tile(dyn, (tile, 1, 1, 1, 1))
        pl = _planner()
        full = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0])
        want = {k: getattr(full, k).copy() for k in ("best_idx", "best_cost", "stats", "winner_len", "winner")}
        for env in (dict(), dict(FOT_GATED=0)):
            with _env(**env):
                for k in (2, 7):
                    res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0], winner_samples=k)
                    assert res.winner.shape == (len(frenet), 15, k)
                    for key in ("best_idx", "stats", "winner_len"):
                        assert np.array_equal(getattr(res, key), want[key]), (env, k, key)
                    assert np.array_equal(res.best_cost.view(np.uint64), want["best_cost"].view(np.uint64))
                    keep = np.arange(k)[None, None, :] < np.minimum(want["winner_len"], k)[:, None, None]
                    assert np.array_equal(np.where(keep, res.winner, 0.0).view(np.uint64),
                                          np.where(keep, want["winner"][:, :, :k], 0.0).view(np.uint64)), (env, k)
                    q0, n = len(frenet) // 3, min(5, len(frenet) - len(frenet) // 3)
                    got = pl.engine.fetch_winners(q0, n)
                    lens = want["winner_len"][q0:q0 + n]
                    assert _same("winner", got, want["winner"][q0:q0 + n], lens), (env, k)
                    series = res.series(int(np.argmax(want["best_idx"] >= 0))) if (want["best_idx"] >= 0).any() else None
                    assert series is None or len(series["x"]) <= k


def test_pair_kernel_shape_limits_and_fallback():
    """fot_sweep_pairs has compile-time shape limits (56 samples per profile, 96 lateral targets, 48 spline knots): at the
    limits it runs, one step beyond them fot_sweep_items takes over -- and either way every candidate's category is the
    oracle's."""
    rng = np.random.default_rng(23)
    k = scenarios.S1_KNOBS
    dyn = scenarios.pedestrian_field(rng, 12, n_steps=60)
    fs = np.array([[4.0, 5.0, 0.2, 0.3, 0.05, 0.0], [6.0, 2.0, -0.5, -0.8, 0.0, 0.02]])
    cases = [
        (dict(k, max_t=5.5, min_t=5.0), scenarios.STRAIGHT_60, 4),                      # 56 samples: the last shape the pair kernel takes
        (dict(k, max_t=5.6, min_t=5.2), scenarios.STRAIGHT_60, 1),                      # 57 samples
        (dict(k, d_road_w=2.7 / 47.5, min_t=4.8), scenarios.STRAIGHT_60, 4),            # 95 lateral targets
        (dict(k, d_road_w=2.7 / 48.5, min_t=4.8), scenarios.STRAIGHT_60, 1),            # 97 lateral targets
        (dict(k, min_t=4.8), scenarios.arc_waypoints(n=48), 4),                         # 48 spline knots
        (dict(k, min_t=4.8), scenarios.arc_waypoints(n=49), 1),                         # 49
    ]
    for knobs, wp, kind in cases:
        pl, orc = _planner(knobs, wp), _oracle(knobs, wp)
        res = pl.plan_batch(fs, 6.0, dynamic_obstacles=np.stack([dyn] * 2), want_candidates=True)
        assert int(pl.engine.lib.fot_last_sweep_kind(pl.engine._h)) == kind, (knobs, kind)
        _check(res, [orc.plan_frenet(tuple(s), np.empty((0, 2)), dyn, 6.0) for s in fs])


def test_long_time_grid_large_upload_matches_the_resident_launch():
    """A time grid of 129 samples is beyond fot_sweep_pairs, so fot_sweep_items runs.  The upload size (1024 queries x
    5 pedestrians x 129 steps, 10.6 MB) and FOT_HOST_CHUNKS cut the batch into query ranges, and the host-pointer call
    may gate the sweep on the upload.  Both host-result calls must return the bits of a plain launch over the resident
    tensor."""
    import torch
    from integrated_path_planning_b200 import DeviceBatch, _lib
    knobs = dict(scenarios.S1_KNOBS, dt=0.05, min_t=6.0, max_t=6.4, d_road_w=0.9, d_t_s=3.0)
    rng = np.random.default_rng(41)
    n = 1024
    frenet = np.stack([rng.uniform(2, 15, n), rng.uniform(1, 7, n), rng.uniform(-1, 1, n), rng.uniform(-1, 1, n),
                       rng.normal(0, 0.2, n), rng.normal(0, 0.05, n)], axis=1)
    dyn = np.stack([scenarios.pedestrian_field(rng, 5, n_steps=129, dt=0.05) for _ in range(n)])
    pl = _planner(knobs)
    assert pl.engine.n_t_max > 128
    batch = DeviceBatch(pl, frenet, 6.0, dyn[:, None], _lib.FOT_DYN_SINGLE)
    batch.launch(None)
    assert int(pl.engine.lib.fot_last_sweep_kind(pl.engine._h)) == 1
    want = {k: v.cpu().numpy() for k, v in batch.out.items()}
    assert len(set(want["best_idx"].tolist())) > 5

    def agree(got, how):
        for k, v in want.items():
            assert _same(k, v, np.asarray(got[k]), want["winner_len"]), (how, k)

    res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn, want_candidates=True)
    assert int(pl.engine.lib.fot_last_sweep_kind(pl.engine._h)) == 1
    agree({k: getattr(res, k) for k in want}, "plan_batch")
    orc = _oracle(knobs)
    _check(res, [orc.plan_frenet(tuple(frenet[i]), np.empty((0, 2)), dyn[i], 6.0) for i in range(3)])
    with _env(FOT_HOST_CHUNKS=3):
        res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn)
    agree({k: getattr(res, k) for k in want}, "FOT_HOST_CHUNKS=3")
    host = {k: torch.full(v.shape, -7, dtype=v.dtype).pin_memory() for k, v in batch.out.items()}
    batch.launch_to_host(host)
    agree({k: v.numpy() for k, v in host.items()}, "launch_to_host")
