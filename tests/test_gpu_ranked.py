"""GPU: ranked alternatives (fot_rank_candidates) -- the k best feasible candidates of every query and their series.

The ranking is held to three yardsticks: the winner of the same launch (rank 0), the per-candidate table of the same
launch sorted on the host by (cost, index), and the NumPy oracle's categories, costs and candidate arrays."""
import ctypes as C

import numpy as np
import pytest

from oracle import frenet_oracle as O
from tests import campaign, runners, scenarios

pytestmark = pytest.mark.gpu


def _planner(knobs=None, wp=scenarios.STRAIGHT_60, **kw):
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    return BatchFrenetPlanner(CubicSpline2D(*wp), **dict(knobs or scenarios.S1_KNOBS), **kw)


@pytest.fixture(scope="module")
def config4():
    import bench
    _, frenet, dyn = bench.make_queries(3000, 512)
    return frenet, dyn


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _host_rank(cat, cost, k):
    """The first k feasible candidates of one table row by (cost, index): category OK, cost below +inf."""
    with np.errstate(invalid="ignore"):
        ok = np.nonzero((cat == 0) & (cost < np.inf))[0]
    idx = ok[np.lexsort((ok, cost[ok]))][:k]
    return idx, cost[idx]


def _assert_ranks_follow_table(res, k, n_cand=None):
    """Every query's ranks are the table's feasible entries in (cost, index) order, padded with -1 / +inf / 0.
    Returns the number of feasible candidates per query."""
    n_q = len(res.best_idx)
    assert res.rank_idx.shape == (n_q, k) and res.rank_cost.shape == (n_q, k)
    n_feasible = np.zeros(n_q, dtype=np.int64)
    bad = []
    for q in range(n_q):
        row = slice(None) if n_cand is None else slice(0, int(n_cand[q]))
        idx, cost = _host_rank(res.cand_cat[q, row], res.cand_cost[q, row], k)
        n = len(idx)
        with np.errstate(invalid="ignore"):
            n_feasible[q] = int(((res.cand_cat[q, row] == 0) & (res.cand_cost[q, row] < np.inf)).sum())
        ok = np.array_equal(res.rank_idx[q, :n], idx) and np.array_equal(_bits(res.rank_cost[q, :n]), _bits(cost))
        ok &= bool(np.all(res.rank_idx[q, n:] == -1) and np.all(np.isposinf(res.rank_cost[q, n:])))
        if res.rank_len is not None:
            ok &= bool(np.all(res.rank_len[q, n:] == 0) and np.all(res.rank_len[q, :n] > 0))
        if not ok:
            bad.append(q)
    assert not bad, (f"{len(bad)} of {n_q} queries rank differently from their table: {bad[:10]}",
                     res.rank_idx[bad[0]], _host_rank(res.cand_cat[bad[0]], res.cand_cost[bad[0]], k)[0])
    return n_feasible


def _assert_rank0_is_winner(res):
    assert np.array_equal(res.rank_idx[:, 0], res.best_idx)
    assert np.array_equal(_bits(res.rank_cost[:, 0]), _bits(res.best_cost))
    assert np.array_equal(res.rank_len[:, 0], res.winner_len)
    for q in np.nonzero(res.best_idx >= 0)[0]:
        n = int(res.winner_len[q])
        assert np.array_equal(_bits(res.rank_series[q, 0, :, :n]), _bits(res.winner[q, :, :n])), q


# ---- 1. rank 0 is the winner; 2. the ranks follow the table, on both sweep kernels ---------------------------
@pytest.mark.parametrize("kernel", ["pairs", "items"])
def test_rank0_is_the_winner_config4(config4, kernel):
    frenet, dyn = config4
    pl = _planner()
    pl.engine
    with runners.fot_env(FOT_SWEEP=kernel):
        res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0], top_k=8, want_candidates=True)
        assert int(pl.engine.lib.fot_last_sweep_kind(pl.engine._h)) == {"pairs": 4, "items": 1}[kernel]
    assert (res.best_idx >= 0).sum() > 100
    _assert_rank0_is_winner(res)
    n_feasible = _assert_ranks_follow_table(res, 8, res.n_cand)
    assert (n_feasible >= 8).sum() > 100
    # every ranked alternative is a feasible candidate of the table with that cost, and the series start at the ego
    for q in np.nonzero(res.best_idx >= 0)[0][:64]:
        for r, a in enumerate(res.alternatives(q)):
            assert res.cand_cat[q, a["index"]] == 0 and a["cost"] == res.cand_cost[q, a["index"]]
            assert a["series"]["s"][0] == frenet[q, 0] and len(a["series"]["x"]) == res.rank_len[q, r]


# ---- 2. the ranks follow the table -------------------------------------------------------------------------------
def test_ranks_follow_table_near_limit_queries():
    """Campaign B: limits through the candidates' range (every category populated) and the stop-distance directive."""
    qs = [campaign.query_b(i) for i in range(campaign.N_B)]
    n_partial = n_none = n_full = 0
    for path in campaign.PATH_NAMES:
        for road in (2.7, 1.1):
            ids = [i for i, q in enumerate(qs) if q["path"] == path and q["road"] == road]
            pl = _planner(campaign.knobs_b(road), campaign.PATHS[path])
            limits = np.stack([pl.resolve_limits(qs[i]["overrides"]) for i in ids])
            msd = np.array([np.nan if qs[i]["msd"] is None else qs[i]["msd"] for i in ids])
            res = pl.plan_batch(np.stack([qs[i]["fs"] for i in ids]), np.array([qs[i]["target"] for i in ids]),
                                dynamic_obstacles=np.stack([qs[i]["dyn"] for i in ids]), limits=limits,
                                max_stop_distance=msd, want_candidates=True, top_k=32)
            _assert_rank0_is_winner(res)
            n = _assert_ranks_follow_table(res, 32, res.n_cand)
            n_none += int((n == 0).sum())
            n_partial += int(((n > 0) & (n < 32)).sum())
            n_full += int((n >= 32).sum())
    # padding: queries without any feasible candidate and queries with fewer than k of them are both present
    assert n_none > 0 and n_partial > 0 and n_full > 0, (n_none, n_partial, n_full)


@pytest.mark.parametrize("variant", [0, 1])
def test_ranks_follow_table_config3(variant):
    """66 563 candidates per query, distribution mode: the selection streams the row from global memory."""
    c = campaign.config3(variant)
    pl = _planner(c["knobs"], c["waypoints"])
    res = pl.plan_batch(c["fs"][None], c["target"], distribution=c["dist"][None], want_candidates=True, top_k=32)
    assert int(res.n_cand[0]) == 66563
    n = _assert_ranks_follow_table(res, 32, res.n_cand)
    _assert_rank0_is_winner(res)
    if variant == 0:                                       # every candidate rejected: all ranks padded
        assert n[0] == 0 and np.all(res.rank_idx == -1) and np.all(np.isposinf(res.rank_cost)) and np.all(res.rank_len == 0)
    else:
        assert n[0] > 1000 and np.all(res.rank_idx[0] >= 0)


def test_ranks_follow_table_budgeted_distribution_with_footprint():
    rng = np.random.default_rng(5)
    n = 24
    knobs = dict(scenarios.S1_KNOBS, chance_epsilon=0.25)
    frenet = np.stack([rng.uniform(1, 10, n), rng.uniform(1, 7, n), rng.uniform(-1, 1, n),
                       rng.uniform(-1, 1, n), rng.normal(0, 0.2, n), rng.normal(0, 0.05, n)], axis=1)
    dists = []
    for i in range(n):
        r = np.random.default_rng(200 + i)
        base = scenarios.pedestrian_field(r, 14, x_range=(0.0, 20.0), y_range=(-5.0, 25.0))
        dists.append(scenarios.sample_distribution(r, base, 12, sigma=0.08))
    pl = _planner(knobs, scenarios.arc_waypoints(), footprint=runners.make_footprint((4.5, 2.0, 3)))
    res = pl.plan_batch(frenet, 6.0, distribution=np.stack(dists), want_candidates=True, top_k=16)
    _assert_rank0_is_winner(res)
    assert _assert_ranks_follow_table(res, 16, res.n_cand).sum() > 0


def test_ranks_follow_table_static_wall_and_per_query_knobs():
    rng = np.random.default_rng(3)
    n = 96
    k = scenarios.S1_KNOBS
    frenet = np.stack([rng.uniform(2, 30, n), rng.uniform(0, 8, n), rng.uniform(-1, 1, n),
                       rng.uniform(-1.5, 1.5, n), rng.normal(0, 0.3, n), rng.normal(0, 0.05, n)], axis=1)
    target = np.tile([6.0, 3.6, 0.0], n // 3)
    limits = np.tile([[k["max_speed"], k["max_accel"], k["max_curvature"], k["max_lat_accel"]],
                      [k["max_speed"] * 0.6, k["max_accel"] * 1.5, k["max_curvature"], k["max_lat_accel"]],
                      [k["max_speed"], k["max_accel"] * 3.0, k["max_curvature"], k["max_lat_accel"] * 2.0]], (n // 3, 1))
    msd = np.where(target == 0.0, 5.0, np.nan)
    dyn = np.stack([scenarios.pedestrian_field(np.random.default_rng(50 + i), 30, x_range=(0.0, 70.0), y_range=(-8.0, 8.0))
                    for i in range(n)])
    pl = _planner(k, scenarios.s_curve_waypoints())
    res = pl.plan_batch(frenet, target, dynamic_obstacles=dyn, static_obstacles=scenarios.wall(x=45.0, half=1.0, n=9),
                        limits=limits, max_stop_distance=msd, want_candidates=True, top_k=32)
    assert res.stats[:, 6].sum() > 0
    _assert_rank0_is_winner(res)
    _assert_ranks_follow_table(res, 32, res.n_cand)


# ---- 3. the oracle ----------------------------------------------------------------------------------------------
# A wall across the road close ahead, with the EMERGENCY acceleration limit: only short horizons stop in time, so the
# brake ladder ranks -- behind 16 grid candidates with the wall at 18 m, and as the winner with the wall at 16 m.
# (In the standard queries the brake candidates are feasible only without obstacles, at rank 869.)
WALL_AHEAD = [scenarios.Query(f"wall_ahead_{x:.0f}", scenarios.S1_KNOBS, scenarios.STRAIGHT_60, (5.0, 0.0, 0.0, 5.0, 0.0),
                              6.0, static=scenarios.wall(x=x), overrides={"max_accel": 6.0}) for x in (16.0, 18.0)]


def test_ranks_and_series_match_the_oracle():
    k = 32
    bad, brake_ranked = [], 0
    for q in scenarios.standard_queries() + WALL_AHEAD:
        orc = runners.oracle_planner(q)
        static = np.empty((0, 2)) if q.static is None else q.static
        ref = orc.plan(q.ego, static, q.dyn, q.target_speed, q.overrides, q.dist, q.max_stop_distance)
        pl = runners.cuda_planner(q)
        alts = pl.plan_alternatives(runners._Ego(*q.ego), static, q.dyn, q.target_speed, q.overrides, q.dist,
                                    q.max_stop_distance, k=k)
        res = pl.last_result
        idx = np.arange(len(ref.categories))
        with np.errstate(invalid="ignore"):
            feasible = idx[(ref.categories == O.CAT_OK) & (ref.costs < np.inf)]
        want = feasible[np.lexsort((feasible, ref.costs[feasible]))][:k]
        got = res.rank_idx[0][res.rank_idx[0] >= 0]
        if not (np.array_equal(got, want) and np.array_equal(_bits(res.rank_cost[0, :len(got)]), _bits(ref.costs[want]))):
            n = min(len(got), len(want))
            bad.append((q.name, len(got), len(want), int((got[:n] != want[:n]).sum()),
                        int((_bits(res.rank_cost[0, :n]) != _bits(ref.costs[want[:n]])).sum())))
            continue
        assert [int(p.cost == c) for p, c in zip(alts, ref.costs[want])] == [1] * len(want), q.name
        kn = orc.k
        n_grid = len(O.horizon_grid(kn)) * len(O.speed_grid(kn, q.target_speed)) * len(O.lateral_grid(kn))
        brake_ranked += int((want >= n_grid).sum())
        for path, i in zip(alts, want):
            cand = orc.last_candidates[int(i)]
            for name in runners.SERIES:
                got_s = np.asarray(getattr(path, name), dtype=float)
                want_s = np.asarray(getattr(cand, name), dtype=float)
                assert got_s.shape == want_s.shape, (q.name, int(i), name, got_s.shape, want_s.shape)
                np.testing.assert_allclose(got_s, want_s, rtol=runners.RTOL, atol=runners.ATOL,
                                           err_msg=f"{q.name} candidate {int(i)} {name}")
    assert not bad, bad
    assert brake_ranked > 0


# ---- 4. padding -------------------------------------------------------------------------------------------------
def test_padding_k_above_candidate_count():
    """One lateral target, one horizon, target speed 0: one candidate without the brake ladder, 1 + n_B with it."""
    knobs = dict(scenarios.S1_KNOBS, min_t=4.0, max_t=4.0, d_road_w=6.0)
    pl = _planner(knobs)
    frenet = np.array([[5.0, 0.05, 0.0, 0.2, 0.0, 0.0],        # too slow for the brake ladder
                       [5.0, 3.0, 0.0, 0.2, 0.0, 0.0]])
    res = pl.plan_batch(frenet, 0.0, want_candidates=True, top_k=32)
    assert res.n_cand[0] == 1 and 1 < res.n_cand[1] < 32
    n = _assert_ranks_follow_table(res, 32, res.n_cand)
    _assert_rank0_is_winner(res)
    assert n[0] <= 1 and n[1] <= res.n_cand[1] and n.sum() > 0
    assert np.all(res.rank_idx[0, 1:] == -1) and np.all(res.rank_idx[1, res.n_cand[1]:] == -1)


def test_padding_non_finite_states():
    """NaN / inf in the Frenet state drops every candidate (tests/test_gpu_edges.py): all ranks padded, and the finite
    neighbour in the same batch ranks as its table says."""
    dyn = scenarios.pedestrian_field(np.random.default_rng(1), 5)
    states = np.array([[5.0, np.nan, 0, 0, 0, 0], [5.0, 5.0, 0.0, np.inf, 0.0, 0.0], [np.nan, 5, 0, 0, 0, 0],
                       [5.0, 5.0, 0.0, 0.1, 0.0, 0.0]])
    res = _planner().plan_batch(states, 6.0, dynamic_obstacles=np.stack([dyn] * 4), want_candidates=True, top_k=8)
    n = _assert_ranks_follow_table(res, 8, res.n_cand)
    _assert_rank0_is_winner(res)
    assert n[:3].tolist() == [0, 0, 0] and n[3] > 0
    assert np.all(res.rank_idx[:3] == -1) and np.all(np.isposinf(res.rank_cost[:3])) and np.all(res.rank_len[:3] == 0)


# ---- 5. the default launch is unchanged ------------------------------------------------------------------------
def test_unranked_launch_unchanged(config4):
    import torch
    from integrated_path_planning_b200 import _lib
    from integrated_path_planning_b200.batch import DeviceBatch
    frenet, dyn = config4
    pl = _planner()
    lib, h = pl.engine.lib, pl.engine._h
    plain = DeviceBatch(pl, frenet, 6.0, dyn, _lib.FOT_DYN_SINGLE)
    plain.launch()
    assert int(lib.fot_last_sweep_kind(h)) == 4 and int(lib.fot_last_pair_features(h)) == 0
    ranked = DeviceBatch(pl, frenet, 6.0, dyn, _lib.FOT_DYN_SINGLE, top_k=8)
    ranked.launch()
    assert int(lib.fot_last_pair_features(h)) == 8                 # the instantiation with per-candidate outputs
    lean = DeviceBatch(pl, frenet, 6.0, dyn, _lib.FOT_DYN_SINGLE, top_k=8, rank_series=False)
    lean.launch()
    plain.launch()
    assert int(lib.fot_last_pair_features(h)) == 0
    torch.cuda.synchronize()
    a, b, c = ({k: v.cpu().numpy() for k, v in x.out.items()} for x in (plain, ranked, lean))
    assert set(a) == {"best_idx", "best_cost", "stats", "winner_len", "winner"}
    assert "rank_len" not in c and "rank_series" not in c
    for x in (b, c):
        for key in ("best_idx", "stats", "winner_len"):
            assert np.array_equal(a[key], x[key]), key
        assert np.array_equal(_bits(a["best_cost"]), _bits(x["best_cost"]))
        for q in np.nonzero(a["best_idx"] >= 0)[0]:
            n = int(a["winner_len"][q])
            assert np.array_equal(_bits(a["winner"][q, :, :n]), _bits(x["winner"][q, :, :n])), q
    assert np.array_equal(b["rank_idx"], c["rank_idx"]) and np.array_equal(_bits(b["rank_cost"]), _bits(c["rank_cost"]))
    host = {k: np.zeros(v.shape, dtype=v.dtype) for k, v in a.items()}
    with pytest.raises(ValueError):
        ranked.launch_to_host(host)


# ---- 6. plan_alternatives against plan() -----------------------------------------------------------------------
def test_plan_alternatives_lock_step_with_plan():
    from integrated_path_planning_b200 import CubicSpline2D, FrenetPlanner
    store = runners.load_golden("closed_loop_s01.npz")
    wp = (store["waypoints_x"], store["waypoints_y"])
    one = FrenetPlanner(CubicSpline2D(*wp), **scenarios.S1_KNOBS)
    alt = FrenetPlanner(CubicSpline2D(*wp), **scenarios.S1_KNOBS)
    n_calls, n_found, n_several = len(store["kept"]), 0, 0
    for j in range(n_calls):
        g = runners.golden_case(store, f"c{j}")
        for pl in (one, alt):                              # the recorded pre-call state (the calls are a subset of the run)
            pl._last_kappa = float(g["last_kappa"])
            if np.isnan(g["prev_s"]):
                if hasattr(pl.converter, "_prev_s"):
                    del pl.converter._prev_s
            else:
                pl.converter._prev_s = float(g["prev_s"])
        ovr = {k: float(v) for k, v in zip(("max_speed", "max_accel", "max_curvature", "max_lat_accel"), g["ovr"])
               if not np.isnan(v)} or None
        msd = None if np.isnan(g["msd"]) else float(g["msd"])
        args = (runners._Ego(*g["ego"]), np.empty((0, 2)), g["dyn"], float(g["target"]), ovr, None, msd)
        path = one.plan(*args)
        paths = alt.plan_alternatives(*args, k=6)
        assert (path is None) == (paths == []), j
        assert one.last_check_stats == alt.last_check_stats, j
        assert one._last_kappa == alt._last_kappa, j
        assert getattr(one.converter, "_prev_s", None) == getattr(alt.converter, "_prev_s", None), j
        if path is None:
            continue
        n_found += 1
        n_several += len(paths) > 1
        costs = [float(p.cost) for p in paths]
        assert len(paths) <= 6 and costs == sorted(costs), j
        assert _bits(paths[0].cost) == _bits(path.cost), j
        for name in runners.SERIES:
            assert np.array_equal(_bits(getattr(paths[0], name)), _bits(getattr(path, name))), (j, name)
            assert type(getattr(paths[0], name)) is type(getattr(path, name)), (j, name)
    assert n_found > 0 and n_several > 0


# ---- 7. argument errors -----------------------------------------------------------------------------------------
def test_rank_candidates_rejects_bad_arguments(config4):
    from integrated_path_planning_b200 import _lib
    from integrated_path_planning_b200.batch import DeviceBatch
    frenet, dyn = config4
    pl = _planner()
    db = DeviceBatch(pl, frenet[:16], 6.0, dyn[:16], _lib.FOT_DYN_SINGLE, top_k=4)
    db.launch()
    eng, r = pl.engine, db.result
    good_len = db.out["rank_len"].cpu().numpy().copy()

    def call(batch=None, ranked=None, stride=None, cat=None):
        eng.rank_device(batch or db.batch, r.cand_cat if cat is None else cat, r.cand_cost,
                        r.cand_stride if stride is None else stride, ranked or db.ranked)

    def ranked(**kw):
        x = _lib.FotRanked.from_buffer_copy(db.ranked)
        for key, v in kw.items():
            setattr(x, key, v)
        return x

    empty = _lib.FotBatch.from_buffer_copy(db.batch)
    empty.n_q = 0
    bad_calls = [dict(ranked=ranked(k=0)), dict(ranked=ranked(k=_lib.FOT_MAX_RANKED + 1)), dict(ranked=ranked(idx=None)),
                 dict(ranked=ranked(cost=None)), dict(ranked=ranked(len=None)), dict(stride=r.cand_stride - 1),
                 dict(batch=empty), dict(cat=0)]
    for kw in bad_calls:
        with pytest.raises(_lib.FotError):
            call(**kw)
    # lengths without series are allowed (ranked(series=None)); they equal the lengths that come with the series
    db.out["rank_len"].fill_(-5)
    call(ranked=ranked(series=None))
    assert np.array_equal(db.out["rank_len"].cpu().numpy(), good_len)
    assert int(C.sizeof(_lib.FotRanked)) == 40
