"""GPU: multi-route batches -- every query planned on its own reference path in one launch (fot_add_route,
fot_set_routes; DESIGN.md section 4h).

The yardstick is a planner created with the query's path alone: a routed query must give its winner index, cost bits,
stats, kept length, series bits and (when requested) per-candidate categories and costs.  A query with a bad route id
comes back blank and leaves its neighbours alone."""
import numpy as np
import pytest

from oracle import frenet_oracle as O
from tests import campaign, runners, scenarios

pytestmark = pytest.mark.gpu

SHORT = [scenarios.STRAIGHT_60, scenarios.s_curve_waypoints(), scenarios.arc_waypoints()]   # <= 48 knots: pair kernel
LONG = SHORT + [campaign.C_PATH]                                                            # 60 knots: fot_sweep_items
N_Q = 48


def _planner(wp, knobs):
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    return BatchFrenetPlanner(CubicSpline2D(*wp), **knobs)


def _routed(paths, knobs):
    from integrated_path_planning_b200 import CubicSpline2D
    pl = _planner(paths[0], knobs)
    for wp in paths[1:]:
        assert pl.add_route(CubicSpline2D(*wp)) == len(pl.routes) - 1
    return pl


def _knobs(mode):
    k = dict(scenarios.S1_KNOBS)
    if mode == "dist":
        k["chance_epsilon"] = 0.1                     # a violation budget of 1 in 10 samples
    if mode == "static_fp":
        k["footprint"] = runners.make_footprint((4.5, 1.9, 3))
    return k


def _queries(mode, n_q=N_Q, seed=7, n_routes=3):
    """(frenet [n_q,6], plan_batch keywords, route [n_q]) of a mixed batch."""
    rng = np.random.default_rng(seed)
    fs = np.stack([campaign.query_b(i)["fs"] for i in range(n_q)])
    fs[:, 0] = rng.uniform(3.0, 40.0, n_q)
    dyn = np.stack([scenarios.pedestrian_field(rng, 6, x_range=(0.0, 50.0)) for _ in range(n_q)])
    kw = dict(target_speed=6.0)
    if mode == "dist":
        kw["distribution"] = np.stack([scenarios.sample_distribution(rng, d, 10) for d in dyn])
    else:
        kw["dynamic_obstacles"] = dyn
    if mode == "static_fp":
        kw["static_obstacles"] = scenarios.wall(x=20.0, half=3.0, n=13)
    route = (np.arange(n_q) * 7 + 3) % n_routes
    return fs, kw, route.astype(np.int64)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _select(kw, rows):
    return {k: (v[rows] if k in ("dynamic_obstacles", "distribution") else v) for k, v in kw.items()}


def _per_route(paths, knobs, fs, kw, route, **run):
    """The yardstick: one planner per path, each planning its own queries."""
    out = {}
    for r, wp in enumerate(paths):
        rows = np.nonzero(route == r)[0]
        if len(rows):
            out[r] = (rows, _planner(wp, knobs).plan_batch(fs[rows], **_select(kw, rows), **run))
    return out


def _assert_same(res, ref, rows, cands=False, ref_rows=None):
    """res's queries `rows` equal ref's `ref_rows` (default: ref's queries 0, 1, ...)."""
    for j, q in zip(range(len(rows)) if ref_rows is None else ref_rows, rows):
        assert res.best_idx[q] == ref.best_idx[j], (q, res.best_idx[q], ref.best_idx[j])
        assert _bits(res.best_cost[q]) == _bits(ref.best_cost[j]), q
        assert np.array_equal(res.stats[q], ref.stats[j]), (q, res.stats[q], ref.stats[j])
        assert res.winner_len[q] == ref.winner_len[j], q
        n = int(res.winner_len[q])
        assert np.array_equal(_bits(res.winner[q, :, :n]), _bits(ref.winner[j, :, :n])), q
        if cands:
            m = int(ref.n_cand[j])
            assert np.array_equal(res.cand_cat[q, :m], ref.cand_cat[j, :m]), q
            assert np.array_equal(_bits(res.cand_cost[q, :m]), _bits(ref.cand_cost[j, :m])), q


def _assert_selections(res, rows, ref, ref_rows):
    """Ranked and weighted outputs of res's queries `rows` equal ref's `ref_rows`: indices, cost bits, kept lengths and
    the kept samples of every series (padding entries write no series row)."""
    for block in ("rank", "w"):
        idx, ridx = getattr(res, block + "_idx")[rows], getattr(ref, block + "_idx")[ref_rows]
        assert np.array_equal(idx, ridx), block
        assert np.array_equal(_bits(getattr(res, block + "_cost")[rows]), _bits(getattr(ref, block + "_cost")[ref_rows]))
        ln, rln = getattr(res, block + "_len")[rows], getattr(ref, block + "_len")[ref_rows]
        assert np.array_equal(ln, rln), block
        ser, rser = getattr(res, block + "_series")[rows], getattr(ref, block + "_series")[ref_rows]
        for q, j in zip(*np.nonzero(idx >= 0)):
            n = int(ln[q, j])
            assert np.array_equal(_bits(ser[q, j, :, :n]), _bits(rser[q, j, :, :n])), (block, q, j)


def _assert_routed(paths, knobs, fs, kw, route, res, **run):
    for rows, ref in _per_route(paths, knobs, fs, kw, route, **run).values():
        _assert_same(res, ref, rows, cands=run.get("want_candidates", False))


# ---- routed equals single-route on every sweep path -------------------------------------------------------------
@pytest.mark.parametrize("mode", ["single", "dist", "static_fp"])
@pytest.mark.parametrize("kernel", ["pairs", "items", "long"])
def test_routed_host_call_equals_single_route(mode, kernel):
    from integrated_path_planning_b200 import _lib
    paths = LONG if kernel == "long" else SHORT
    knobs = _knobs(mode)
    pl = _routed(paths, knobs)
    fs, kw, route = _queries(mode, n_routes=len(paths))
    with runners.fot_env(FOT_SWEEP="items" if kernel == "items" else "0"):
        runners.reload_options()
        res = pl.plan_batch(fs, **kw, route=route, want_candidates=True)
        kind = pl.engine.lib.fot_last_sweep_kind(pl.engine._h)
        feat = pl.engine.lib.fot_last_pair_features(pl.engine._h)
    runners.reload_options()
    if kernel == "pairs":
        assert kind == 4
        want = {"single": 32 | 8, "dist": 32 | 31, "static_fp": 32 | 31}[mode]   # + per-candidate outputs
        assert feat == want, (feat, want)
    else:
        assert kind == 1 and feat == -1
    _assert_routed(paths, knobs, fs, kw, route, res, want_candidates=True)
    assert _lib.FOT_ABI_MINOR == 1


def test_routed_campaign_shape_picks_the_routed_campaign_kernel():
    pl = _routed(SHORT, _knobs("single"))
    fs, kw, route = _queries("single")
    res = pl.plan_batch(fs, **kw, route=route)
    assert pl.engine.lib.fot_last_sweep_kind(pl.engine._h) == 4
    assert pl.engine.lib.fot_last_pair_features(pl.engine._h) == 32
    _assert_routed(SHORT, _knobs("single"), fs, kw, route, res)


def test_routed_gated_host_call():
    """The host-pointer call in several query ranges, gated on the obstacle upload: the route array is offset with
    every range."""
    pl = _routed(SHORT, _knobs("single"))
    fs, kw, route = _queries("single", n_q=600)
    with runners.fot_env(FOT_HOST_CHUNKS=4):
        runners.reload_options()
        res = pl.plan_batch(fs, **kw, route=route)
    runners.reload_options()
    _assert_routed(SHORT, _knobs("single"), fs, kw, route, res)


@pytest.mark.parametrize("paths", ["short", "long"])
def test_routed_device_and_launch_to_host(paths):
    import torch
    from integrated_path_planning_b200 import DeviceBatch, _lib
    paths = SHORT if paths == "short" else LONG
    knobs = _knobs("single")
    pl = _routed(paths, knobs)
    fs, kw, route = _queries("single", n_q=300, n_routes=len(paths))
    dyn = kw["dynamic_obstacles"][:, None]
    db = DeviceBatch(pl, fs, 6.0, dyn, _lib.FOT_DYN_SINGLE, route=route)
    db.launch()
    res = db.sweep_result()
    _assert_routed(paths, knobs, fs, kw, route, res)
    host = {k: torch.empty(v.shape if k != "winner" else (len(fs), _lib.FOT_N_SERIES, 2), dtype=v.dtype).pin_memory()
            for k, v in db.out.items()}
    db.launch_to_host(host, winner_samples=2)
    for k in ("best_idx", "best_cost", "stats", "winner_len"):
        assert np.array_equal(host[k].numpy().view(np.uint8), getattr(res, k).view(np.uint8)), k
    for q in np.nonzero(res.best_idx >= 0)[0]:                           # rows without a winner are not written
        n = min(2, int(res.winner_len[q]))
        assert np.array_equal(_bits(host["winner"].numpy()[q, :, :n]), _bits(res.winner[q, :, :n])), q


# ---- bad route ids ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("paths", ["short", "long"])
def test_bad_route_id_is_blank_and_leaves_neighbours_alone(paths):
    import torch
    from integrated_path_planning_b200 import DeviceBatch, _lib
    paths = SHORT if paths == "short" else LONG
    pl = _routed(paths, _knobs("single"))
    fs, kw, route = _queries("single", n_routes=len(paths))
    dyn = kw["dynamic_obstacles"][:, None]
    w = np.array([[1.0, 1.0, 1.0, 1.0, 1.0, 1.0], [0.5, 2.0, 1.0, 3.0, 1.0, 0.7]])
    good = DeviceBatch(pl, fs, 6.0, dyn, _lib.FOT_DYN_SINGLE, route=route, top_k=8, cost_weights=w)
    good.launch()
    ref = good.sweep_result(want_candidates=True)
    bad = DeviceBatch(pl, fs, 6.0, dyn, _lib.FOT_DYN_SINGLE, route=route, top_k=8, cost_weights=w)
    rows = [3, 17, 30]
    bad.t["route"][torch.tensor(rows, device=bad.t["route"].device)] = torch.tensor([len(paths), -1, 1 << 20],
                                                                                  dtype=torch.int32, device=bad.t["route"].device)
    bad.launch()
    res = bad.sweep_result(want_candidates=True)
    assert np.all(res.best_idx[rows] == -1) and np.all(np.isposinf(res.best_cost[rows]))
    assert np.all(res.stats[rows] == 0) and np.all(res.winner_len[rows] == 0)
    assert np.all(res.rank_idx[rows] == -1) and np.all(res.w_idx[rows] == -1)
    assert np.all(res.cand_cat[rows] == _lib.CAT_DROP + 1)               # never written
    keep = np.setdiff1d(np.arange(len(fs)), rows)
    _assert_same(res, ref, keep, ref_rows=keep)
    _assert_selections(res, keep, ref, keep)


# ---- selections, route 0 and the search --------------------------------------------------------------------------
def test_routed_top_k_and_cost_weights_equal_per_route_planners():
    knobs = _knobs("single")
    pl = _routed(SHORT, knobs)
    fs, kw, route = _queries("single")
    w = np.array([[1.0, 1.0, 1.0, 1.0, 1.0, 1.0], [0.2, 1.5, 4.0, 0.5, 1.0, 2.0], [3.0, 0.1, 0.3, 2.0, 0.5, 1.0]])
    run = dict(top_k=8, cost_weights=w, want_candidates=True)
    res = pl.plan_batch(fs, **kw, route=route, **run)
    for rows, ref in _per_route(SHORT, knobs, fs, kw, route, **run).values():
        _assert_same(res, ref, rows, cands=True)
        _assert_selections(res, rows, ref, np.arange(len(rows)))


def test_route_zero_and_no_route_equal_an_unrouted_planner():
    knobs = _knobs("single")
    fs, kw, _ = _queries("single")
    plain = _planner(SHORT[0], knobs).plan_batch(fs, **kw, want_candidates=True)
    pl = _routed(SHORT, knobs)
    for route in (None, 0, np.zeros(len(fs), dtype=np.int32)):
        res = pl.plan_batch(fs, **kw, route=route, want_candidates=True)
        _assert_same(res, plain, np.arange(len(fs)), cands=True)


def test_routed_nearest_search_equals_per_route_engines():
    rng = np.random.default_rng(11)
    pl = _routed(LONG, _knobs("single"))
    m = 400
    route = rng.integers(0, len(LONG), m)
    x, y = rng.uniform(-5.0, 80.0, m), rng.uniform(-10.0, 20.0, m)
    prev = np.where(rng.uniform(size=m) < 0.5, rng.uniform(0.0, 60.0, m), np.nan)
    s, st = pl.engine.nearest_s(x, y, prev, route=route)
    for r, wp in enumerate(LONG):
        rows = np.nonzero(route == r)[0]
        s_r, st_r = _planner(wp, _knobs("single")).engine.nearest_s(x[rows], y[rows], prev[rows])
        assert np.array_equal(_bits(s[rows]), _bits(s_r)) and np.array_equal(st[rows], st_r), r


def test_routed_plan_batch_from_ego_equals_per_route_planners():
    from integrated_path_planning_b200.frenet_host import BatchCoordinateConverter, RoutedCoordinateConverter
    rng = np.random.default_rng(5)
    knobs = _knobs("single")
    pl = _routed(SHORT, knobs)
    n_q = 60
    route = rng.integers(0, len(SHORT), n_q)
    ego = np.stack([rng.uniform(2, 30, n_q), rng.uniform(-1, 3, n_q), rng.normal(0, 0.1, n_q), rng.uniform(0, 8, n_q),
                    rng.uniform(-1, 1, n_q)], axis=1)
    ego[7] = (np.nan, 0.0, 0.0, 1.0, 0.0)                                  # rows the device search cannot certify
    ego[11] = (1e6, -1e6, 0.0, 1.0, 0.0)
    dyn = np.stack([scenarios.pedestrian_field(rng, 6) for _ in range(n_q)])
    conv = RoutedCoordinateConverter(pl.routes, route, engine=pl.engine)
    res, ok = pl.plan_batch_from_ego(ego, 6.0, converter=conv, dynamic_obstacles=dyn, route=route)
    res2, ok2 = pl.plan_batch_from_ego(ego, 6.0, converter=conv, dynamic_obstacles=dyn, route=route)   # warm caches
    dev = host = 0
    for r, wp in enumerate(SHORT):
        rows = np.nonzero(route == r)[0]
        one = _planner(wp, knobs)
        c = BatchCoordinateConverter(one.csp, len(rows), engine=one.engine)
        ref, ok_r = one.plan_batch_from_ego(ego[rows], 6.0, converter=c, dynamic_obstacles=dyn[rows])
        ref2, ok2_r = one.plan_batch_from_ego(ego[rows], 6.0, converter=c, dynamic_obstacles=dyn[rows])
        assert np.array_equal(ok[rows], ok_r) and np.array_equal(ok2[rows], ok2_r)
        _assert_same(res, ref, rows)
        _assert_same(res2, ref2, rows)
        assert np.array_equal(_bits(conv.prev_s[rows]), _bits(c.prev_s))
        dev, host = dev + c.device_rows, host + c.host_rows
    assert (conv.device_rows, conv.host_rows) == (dev, host)


# ---- against the oracle -------------------------------------------------------------------------------------------
def test_routed_queries_match_the_oracle():
    knobs = _knobs("single")
    pl = _routed(LONG, knobs)
    fs, kw, route = _queries("single", n_q=16, n_routes=len(LONG))
    res = pl.plan_batch(fs, **kw, route=route, want_candidates=True)
    kn = O.Knobs(**scenarios.S1_KNOBS)
    for q in range(len(fs)):
        ref = O.OraclePlanner(O.Spline2D(*LONG[route[q]]), kn).plan_frenet(fs[q], np.empty((0, 2)),
                                                                           kw["dynamic_obstacles"][q], 6.0)
        n_c = len(ref.categories)
        assert int(res.n_cand[q]) == n_c
        assert np.array_equal(res.cand_cat[q, :n_c].astype(np.int8), ref.categories), q
        np.testing.assert_allclose(res.cand_cost[q, :n_c], ref.costs, rtol=1e-9, atol=0)
        assert int(res.best_idx[q]) == ref.best_index, q
        from integrated_path_planning_b200 import _lib
        for key, v in ref.stats.items():
            assert int(res.stats[q, _lib.STAT_KEYS.index(key)]) == v, (q, key)
        if ref.best_index >= 0:
            np.testing.assert_allclose(res.best_cost[q], ref.cost, rtol=1e-9, atol=0)
            got = res.series(q)
            for name, want in ref.arrays.items():
                np.testing.assert_allclose(got[name], want, rtol=1e-9, atol=1e-9, err_msg=f"{q} {name}")


# ---- the remaining routed instantiations ---------------------------------------------------------------------------
def test_routed_static_only_runs_the_routed_static_kernel():
    """Static obstacles, one circle, no per-candidate outputs: PAIR_ROUTES | PAIR_STATIC."""
    knobs = _knobs("single")
    pl = _routed(SHORT, knobs)
    fs, kw, route = _queries("single")
    kw["static_obstacles"] = scenarios.wall(x=20.0, half=3.0, n=13)
    res = pl.plan_batch(fs, **kw, route=route)
    assert pl.engine.lib.fot_last_sweep_kind(pl.engine._h) == 4
    assert pl.engine.lib.fot_last_pair_features(pl.engine._h) == 32 | 1
    _assert_routed(SHORT, knobs, fs, kw, route, res)


def test_routed_items_kernel_with_tables_in_global_memory():
    """A route of 140 knots: fot_sweep_items keeps the tables out of shared memory (spline_smem 0, nx > 128) and reads
    each query's route from the global table blob."""
    knobs = _knobs("single")
    paths = SHORT + [scenarios.s_curve_waypoints(length=260.0, amp=3.0, n=140)]
    pl = _routed(paths, knobs)
    fs, kw, route = _queries("single", n_routes=len(paths))
    res = pl.plan_batch(fs, **kw, route=route, want_candidates=True)
    assert pl.engine.lib.fot_last_sweep_kind(pl.engine._h) == 1
    _assert_routed(paths, knobs, fs, kw, route, res, want_candidates=True)


def test_from_ego_refuses_a_converter_on_other_routes():
    from integrated_path_planning_b200.frenet_host import BatchCoordinateConverter, RoutedCoordinateConverter
    pl = _routed(SHORT, _knobs("single"))
    ego = np.tile([5.0, 0.5, 0.0, 3.0, 0.0], (4, 1))
    route = np.array([0, 1, 2, 1])
    with pytest.raises(ValueError):
        pl.plan_batch_from_ego(ego, 6.0, converter=BatchCoordinateConverter(pl.csp, 4, engine=pl.engine), route=route)
    with pytest.raises(ValueError):
        pl.plan_batch_from_ego(ego, 6.0, converter=RoutedCoordinateConverter(pl.routes, [0, 1, 2, 2]), route=route)
    with pytest.raises(ValueError):
        pl.plan_batch_from_ego(ego, 6.0, converter=RoutedCoordinateConverter(pl.routes, route))   # no route: route 0


# ---- closed loop: N simulations over three routes = three single-route loops --------------------------------------
def _closed_loop_setup():
    from integrated_path_planning_b200 import CubicSpline2D
    z, z3 = runners.load_golden("rollout_s01.npz"), runners.load_golden("rollout_s03.npz")
    knobs = {k[5:]: float(z[k]) for k in z.files if k.startswith("knob/")}
    paths = [(z["v0/wx"], z["v0/wy"]), (z3["v0/wx"], z3["v0/wy"]), scenarios.s_curve_waypoints(length=80.0, amp=3.0, n=20)]
    starts = []
    for wx, wy in paths:                                   # on the path's first point, heading along it, at 5 m/s
        sp = CubicSpline2D(list(wx), list(wy))
        x, y = sp.calc_position(0.0)
        starts.append([float(x), float(y), float(sp.calc_yaw(0.0)), 5.0, 0.0])
    route = np.array([0, 1, 2, 0, 1, 2])
    tracks = np.stack([z[f"v{i}/traj"] for i in (0, 1, 2, 3, 0, 1)])
    ego0 = np.array([starts[r] for r in route])
    return knobs, paths, route, tracks, ego0


def test_closed_loop_over_three_routes_equals_single_route_loops(tmp_path):
    import os
    from integrated_path_planning_b200.rollout import BatchedClosedLoop
    knobs, paths, route, tracks, ego0 = _closed_loop_setup()
    n_steps = 160
    sim = BatchedClosedLoop(paths[0][0], paths[0][1], knobs, tracks, ego0, routes=paths[1:], route=route, record=True)
    sim.warmup()
    out = sim.run(n_steps)
    assert sim.planner.engine.lib.fot_last_pair_features(sim.planner.engine._h) & 32
    for r, (wx, wy) in enumerate(paths):
        rows = np.nonzero(route == r)[0]
        one = BatchedClosedLoop(wx, wy, knobs, tracks[rows], ego0[rows], record=True)
        one.warmup()
        ref = one.run(n_steps)
        for key in ("ego", "fsm", "found", "calls", "steps", "reason"):
            a, b = out[key][rows], ref[key]
            # steps after a simulation ended are NaN in the ego history (BatchedClosedLoop.run)
            same = list(a) == list(b) if a.dtype == object else np.array_equal(a, b, equal_nan=a.dtype.kind == "f")
            assert same, (r, key)
        # the result files of the route's first simulation: trajectory.npz and the metric files, byte for byte but
        # for the four wall-clock columns (each driver's own timing)
        d_routed, d_one = str(tmp_path / f"routed{r}"), str(tmp_path / f"one{r}")
        sim.save_results(int(rows[0]), d_routed)
        one.save_results(0, d_one)
        za, zb = np.load(os.path.join(d_routed, "trajectory.npz"), allow_pickle=True), \
            np.load(os.path.join(d_one, "trajectory.npz"), allow_pickle=True)
        assert za.files == zb.files
        for f in za.files:
            a, b = za[f], zb[f]
            if a.dtype == object:
                assert len(a) == len(b) and all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(a, b)), (r, f)
            else:
                assert np.array_equal(a, b), (r, f)
        clock = ("avg_prediction_time", "max_prediction_time", "avg_planning_time", "max_planning_time")
        for name in ("metrics_summary.csv", "metrics_report.txt"):
            la = [l for l in open(os.path.join(d_routed, name)).read().splitlines() if not any(c in l for c in clock)]
            lb = [l for l in open(os.path.join(d_one, name)).read().splitlines() if not any(c in l for c in clock)]
            if name.endswith(".csv"):                     # one header row, one value row: drop the clock columns
                ha, va = (row.split(",") for row in open(os.path.join(d_routed, name)).read().splitlines()[:2])
                hb, vb = (row.split(",") for row in open(os.path.join(d_one, name)).read().splitlines()[:2])
                assert ha == hb
                keep = [i for i, h in enumerate(ha) if h not in clock]
                assert [va[i] for i in keep] == [vb[i] for i in keep], (r, name)
            else:
                assert la == lb, (r, name)
