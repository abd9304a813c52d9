"""GPU: trajectory assessment (fot_assess_trajectories) against its NumPy restatement (tests/assess_oracle.py) on the
reference's own candidate positions, on the library's own winners and ranked alternatives, against another obstacle
field, and at the size limits."""
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import frenet_oracle as O
from tests import assess_oracle as AO
from tests import campaign, runners, scenarios

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _oracle_cands(q: scenarios.Query):
    """The oracle planner's candidates of query q with their global positions (keep > 0 after to_global)."""
    pl = runners.oracle_planner(q)
    static = np.empty((0, 2)) if q.static is None else q.static
    pl.plan(q.ego, static, q.dyn, q.target_speed, q.overrides, q.dist, q.max_stop_distance)
    return pl, [c for c in pl.last_candidates if c.keep > 0]


def _assess_all(pl, cands, static, dyn, dist, r2=None):
    """FrenetPlanner.assess over every candidate, 256 per call."""
    out = []
    for lo in range(0, len(cands), 256):
        res = pl.assess(cands[lo:lo + 256], static, dyn, dist, r2=r2)
        out.extend({k: v[j] for k, v in res.items()} for j in range(len(res["dyn_min"])))
    return out


def _check_against_oracle(kn, dt, cands, got, static, field, r2, exact):
    offsets = kn.footprint_offsets
    bad = []
    for c, g in zip(cands, got):
        ref = AO.assess_trajectory(c.t, c.x, c.y, c.yaw, dt, static=static, dyn=field, r2=r2, offsets=offsets)
        if exact:
            ok = np.array_equal(_bits(g["dyn_min"]), _bits(ref["dyn_min"])) and \
                np.array_equal(_bits(g["static_min"]), _bits(ref["static_min"]))
            ok &= np.array_equal(g["dyn_at"], ref["dyn_at"]) and np.array_equal(g["static_at"], ref["static_at"])
        else:
            ok = bool(np.isclose(g["dyn_min"], ref["dyn_min"], rtol=1e-12, atol=1e-12) or
                      g["dyn_min"] == ref["dyn_min"])
            ok &= bool(np.isclose(g["static_min"], ref["static_min"], rtol=1e-12, atol=1e-12) or
                       g["static_min"] == ref["static_min"])
        for name in ("dyn_hits", "first_hit", "static_hit"):
            ok &= np.array_equal(g[name], ref[name])
        if not ok:
            bad.append((g, ref))
    assert not bad, (f"{len(bad)} of {len(cands)} differ", bad[0])


# ---- 1. the reference's own positions: standard queries (every branch, footprint, distribution, wall, short T_obs,
#         NaN pedestrian, empty field, brake ladder) and near-limit campaign B -----------------------------------------
@pytest.mark.parametrize("q", scenarios.standard_queries(), ids=lambda q: q.name)
def test_standard_queries_against_oracle(q):
    opl, cands = _oracle_cands(q)
    kn = opl.k
    pl = runners.cuda_planner(q)
    static = np.empty((0, 2)) if q.static is None else q.static
    dist = q.dist
    field = dist if dist is not None else (None if q.dyn is None else q.dyn[None])
    own = pl.engine.own_radii(2 if dist is not None else 1)
    extra = np.array([[own[0, 0] * 4.0, own[0, 1] * 0.25], [0.0, 0.0], [1.0, 9.0]])
    got = _assess_all(pl, cands, static, q.dyn, dist, r2=np.concatenate([own, extra]))
    r2 = np.concatenate([own, extra])
    _check_against_oracle(kn, kn.dt, cands, got, static, field, r2, exact=kn.footprint_offsets is None)
    # the verdict under the planner's own pair is the reference's collision test, candidate by candidate
    verdicts = _assess_all(pl, cands, static, q.dyn, dist)
    ref = [O.collision_free(kn, c, static if len(static) else None, q.dyn, dist) for c in cands]
    assert [bool(v["collision_free"]) for v in verdicts] == ref


def test_standard_queries_cover_both_verdicts_and_brake_candidates():
    n_free = n_coll = n_brake = 0
    for q in scenarios.standard_queries():
        opl, cands = _oracle_cands(q)
        static = None if q.static is None else q.static
        for c in cands:
            if O.collision_free(opl.k, c, static, q.dyn, q.dist):
                n_free += 1
            else:
                n_coll += 1
            n_brake += int(len(c.t) > 1 and c.s_d[-1] == 0.0 and c.s[-1] == c.s[-2])
    assert n_free > 100 and n_coll > 100 and n_brake > 0


@pytest.mark.parametrize("i", range(0, 42, 3))
def test_campaign_b_against_oracle(i):
    b = campaign.query_b(i)
    kn = O.Knobs(**campaign.knobs_b(b["road"]))
    opl = O.OraclePlanner(O.Spline2D(*campaign.PATHS[b["path"]]), kn)
    opl.plan_frenet(b["fs"], None, b["dyn"], b["target"], b["overrides"], None, b["msd"])
    cands = [c for c in opl.last_candidates if c.keep > 0]
    from integrated_path_planning_b200 import CubicSpline2D, FrenetPlanner
    pl = FrenetPlanner(CubicSpline2D(*campaign.PATHS[b["path"]]), **campaign.knobs_b(b["road"]))
    got = _assess_all(pl, cands, None, b["dyn"], None)
    _check_against_oracle(kn, kn.dt, cands, got, None, b["dyn"][None], pl.engine.own_radii(1), exact=True)
    assert [bool(g["collision_free"]) for g in got] == [O.collision_free(kn, c, None, b["dyn"], None) for c in cands]


def test_inf_steps_and_per_query_static_points():
    """inf steps are entries, never hits; NaN anywhere drops a pedestrian; per-query static points."""
    rng = np.random.default_rng(3)
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    pl = BatchFrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    n_q = 6
    frenet = np.zeros((n_q, 6))
    frenet[:, 0], frenet[:, 1] = rng.uniform(3, 10, n_q), rng.uniform(2, 6, n_q)
    dyn = np.stack([scenarios.pedestrian_field(rng, 8) for _ in range(n_q)])
    dyn[0, 1, 5:] = np.inf
    dyn[1, 2, 7] = (np.nan, 1.0)
    dyn[2, :, :, 1] = np.inf
    static = np.stack([scenarios.wall(x=30.0 + 3 * q, n=9) for q in range(n_q)])
    res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn, static_obstacles=static, assess=True,
                        assess_r2=[[4.0, 4.0], [25.0, 100.0]])
    for q in range(n_q):
        a = res.assessment(q)
        if res.best_idx[q] < 0:
            assert a["dyn_min"][0] == np.inf and a["first_hit"][0].tolist() == [-1, -1]
            continue
        w = res.series(q)
        ref = AO.assess_trajectory(w["t"], w["x"], w["y"], w["yaw"], pl.dt, static=static[q],
                                   dyn=dyn[q][None], r2=[[4.0, 4.0], [25.0, 100.0]])
        assert _bits(a["dyn_min"][0]) == _bits(ref["dyn_min"]) and _bits(a["static_min"][0]) == _bits(ref["static_min"])
        for name in ("dyn_at", "static_at", "dyn_hits", "first_hit", "static_hit"):
            assert np.array_equal(a[name][0], ref[name]), (q, name, a[name][0], ref[name])


# ---- 2. the library's own outputs: every winner and ranked alternative is collision-free under the own pair --------
@pytest.fixture(scope="module")
def config4():
    import bench
    _, frenet, dyn = bench.make_queries(3000, 512)
    return frenet, dyn


@pytest.mark.parametrize("kernel", ["pairs", "items"])
def test_winners_and_ranks_collision_free_config4(config4, kernel):
    frenet, dyn = config4
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    pl = BatchFrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    pl.engine
    with runners.fot_env(FOT_SWEEP=kernel):
        res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0], top_k=8, assess=True)
    assert res.assessed["dyn_min"].shape == (512, 8) and res.assessed["dyn_hits"].shape == (512, 8, 1)
    has = res.rank_idx >= 0
    assert has.sum() > 512 and (~has).sum() > 0
    assert np.all(res.assessed["dyn_hits"][has][:, 0] == 0) and np.all(res.assessed["static_hit"][has] == 0)
    assert np.all(res.assessed["first_hit"][has] == -1)
    assert np.all(res.assessed["dyn_min"][has] * res.assessed["dyn_min"][has] > pl.engine.collide_r2_single * (1 - 1e-12))
    # padded ranks come back blank
    assert np.all(np.isposinf(res.assessed["dyn_min"][~has])) and np.all(res.assessed["dyn_at"][~has] == -1)
    assert np.all(res.assessed["dyn_hits"][~has] == 0) and np.all(res.assessed["first_hit"][~has] == -1)
    # bit for bit the restatement on the returned series (a sample of queries)
    for q in range(0, 512, 37):
        for r in range(8):
            if res.rank_idx[q, r] < 0:
                continue
            n = int(res.rank_len[q, r])
            s = res.rank_series[q, r]
            ref = AO.assess_trajectory(s[0, :n], s[9, :n], s[10, :n], s[11, :n], pl.dt, dyn=dyn[q, 0][None],
                                       r2=pl.engine.own_radii(1))
            assert _bits(res.assessed["dyn_min"][q, r]) == _bits(ref["dyn_min"]) and np.array_equal(res.assessed["dyn_at"][q, r], ref["dyn_at"])


def test_winner_only_matches_rank0(config4):
    frenet, dyn = config4
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    pl = BatchFrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    a = pl.plan_batch(frenet[:128], 6.0, dynamic_obstacles=dyn[:128, 0], assess=True)
    b = pl.plan_batch(frenet[:128], 6.0, dynamic_obstacles=dyn[:128, 0], top_k=3, assess=True)
    assert a.assessed["dyn_min"].shape == (128, 1)
    assert np.array_equal(_bits(a.assessed["dyn_min"][:, 0]), _bits(b.assessed["dyn_min"][:, 0]))
    assert np.array_equal(a.assessed["dyn_at"][:, 0], b.assessed["dyn_at"][:, 0])
    plain = pl.plan_batch(frenet[:128], 6.0, dynamic_obstacles=dyn[:128, 0])
    assert np.array_equal(plain.best_idx, a.best_idx) and np.array_equal(plain.winner_len, a.winner_len)
    for q in np.nonzero(a.best_idx >= 0)[0]:                          # samples past winner_len are never written
        n = int(a.winner_len[q])
        assert np.array_equal(_bits(plain.winner[q, :, :n]), _bits(a.winner[q, :, :n])), q


@pytest.mark.parametrize("name", ["single", "footprint", "distribution"])
def test_collision_boundary_scenes_winners_are_free(name):
    """The scenes of test_gpu_collision_boundary (obstacles a hair inside and outside the collision radius): every
    winner and ranked alternative is collision-free under the handle's own pair."""
    from tests import test_gpu_collision_boundary as CB
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    names = [k for k in CB.SETUPS if (name == "footprint") == bool(CB.SETUPS[k].footprint) and
             (name == "distribution") == bool(CB.SETUPS[k].dist_s)]
    assert names
    for key in names:
        s = CB.SETUPS[key]
        frenet, dyn, stat = CB.batch(key)
        pl = BatchFrenetPlanner(CubicSpline2D(*s.wp), footprint=runners.make_footprint(s.footprint), **s.knobs)
        kw = dict(distribution=dyn) if s.dist_s else dict(dynamic_obstacles=dyn[:, 0])
        res = pl.plan_batch(frenet, s.target_speed, static_obstacles=stat, top_k=4, assess=True, **kw)
        has = res.rank_idx >= 0
        assert has.any(), key
        allowed = int(np.floor(pl.chance_epsilon * dyn.shape[1])) if s.dist_s else 0
        assert np.all(res.assessed["dyn_hits"][has][:, 0] <= allowed) and np.all(res.assessed["static_hit"][has][:, 0] == 0), key
        assert np.all(np.isposinf(res.assessed["dyn_min"][~has])) and np.all(res.assessed["first_hit"][~has] == -1), key


def test_routed_batch_matches_per_route_planners(config4):
    frenet, dyn = config4
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    paths = [scenarios.STRAIGHT_60, scenarios.s_curve_waypoints()]
    pl = BatchFrenetPlanner(CubicSpline2D(*paths[0]), **scenarios.S1_KNOBS)
    pl.add_route(CubicSpline2D(*paths[1]))
    route = np.arange(64) % 2
    res = pl.plan_batch(frenet[:64], 6.0, dynamic_obstacles=dyn[:64, 0], route=route, top_k=2, assess=True)
    for rid, wp in enumerate(paths):
        one = BatchFrenetPlanner(CubicSpline2D(*wp), **scenarios.S1_KNOBS)
        sel = np.nonzero(route == rid)[0]
        ref = one.plan_batch(frenet[sel], 6.0, dynamic_obstacles=dyn[sel, 0], top_k=2, assess=True)
        for name in ("dyn_min", "static_min"):
            assert np.array_equal(_bits(res.assessed[name][sel]), _bits(ref.assessed[name]))
        for name in ("dyn_at", "static_at", "dyn_hits", "first_hit", "static_hit"):
            assert np.array_equal(res.assessed[name][sel], ref.assessed[name])


def test_launch_to_host_refuses_an_assessed_batch(config4):
    frenet, dyn = config4
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D, DeviceBatch
    pl = BatchFrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    db = DeviceBatch(pl, frenet[:4], 6.0, dyn[:4], 1, assess=True)
    with pytest.raises(ValueError, match="assess"):
        db.launch_to_host({})


# ---- 3. another field: planned on the representative sample, assessed against the whole sample set ------------------
def test_representative_plan_against_the_sample_set():
    rng = np.random.default_rng(21)
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    k = dict(scenarios.S1_KNOBS, chance_epsilon=0.2)
    pl = BatchFrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **k)
    n_q, S = 48, 20
    frenet = np.zeros((n_q, 6))
    frenet[:, 0], frenet[:, 1], frenet[:, 3] = rng.uniform(3, 10, n_q), rng.uniform(2, 6, n_q), rng.uniform(-1, 1, n_q)
    base = np.stack([scenarios.pedestrian_field(rng, 12, x_range=(5.0, 30.0), y_range=(-3.0, 3.0)) for _ in range(n_q)])
    dist = np.stack([scenarios.sample_distribution(rng, base[q], S, sigma=0.15) for q in range(n_q)])
    rep = dist[:, 0]
    res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=rep, assess=True, assess_obstacles=dist)
    own = pl.engine.own_radii(2)
    n_hit = 0
    for q in range(n_q):
        a = res.assessment(q)
        if res.best_idx[q] < 0:
            assert a["dyn_min"][0] == np.inf
            continue
        w = res.series(q)
        ref = AO.assess_trajectory(w["t"], w["x"], w["y"], w["yaw"], pl.dt, dyn=dist[q], r2=own)
        assert _bits(a["dyn_min"][0]) == _bits(ref["dyn_min"]) and np.array_equal(a["dyn_at"][0], ref["dyn_at"])
        assert np.array_equal(a["dyn_hits"][0], ref["dyn_hits"]) and np.array_equal(a["first_hit"][0], ref["first_hit"])
        n_hit += int(ref["dyn_hits"][0] > 0)
    assert n_hit > 0                                                   # the sample set is a different field


# ---- 4. sizes: m = 256, n_t = 320, 8 circles; S*P above 32768 --------------------------------------------------------
def _footprint(n):
    return runners.make_footprint((4.5, 2.0, n))


def test_size_limits_m256_nt320_eight_circles():
    rng = np.random.default_rng(5)
    from integrated_path_planning_b200 import CubicSpline2D, FrenetPlanner
    fp = _footprint(8)
    pl = FrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), footprint=fp, **scenarios.S1_KNOBS)
    paths = []
    for j in range(256):
        n = 320 if j % 5 == 0 else int(rng.integers(0, 321))
        t = np.arange(n) * pl.dt
        paths.append(SimpleNamespace(t=t, x=rng.uniform(0, 40, n), y=rng.uniform(-5, 5, n), yaw=rng.uniform(-3, 3, n)))
    dist = rng.uniform(-5, 45, size=(3, 4, 330, 2))
    static = rng.uniform(-5, 45, size=(7, 2))
    r2 = np.array([[1.0, 1.0], [0.25, 4.0], [9.0, 0.01]])
    got = pl.assess(paths, static, None, dist, r2=r2)
    for j in list(range(0, 256, 17)) + [255]:
        p = paths[j]
        ref = AO.assess_trajectory(p.t, p.x, p.y, p.yaw, pl.dt, static=static, dyn=dist, r2=r2, offsets=fp.offsets)
        assert np.isclose(got["dyn_min"][j], ref["dyn_min"], rtol=1e-12) or got["dyn_min"][j] == ref["dyn_min"]
        assert np.isclose(got["static_min"][j], ref["static_min"], rtol=1e-12) or got["static_min"][j] == ref["static_min"]
        for name in ("dyn_at", "static_at", "dyn_hits", "first_hit", "static_hit"):
            assert np.array_equal(got[name][j], ref[name]), (j, name)


def test_size_sp_above_32768():
    rng = np.random.default_rng(6)
    from integrated_path_planning_b200 import CubicSpline2D, FrenetPlanner
    pl = FrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    S, P, T = 3, 11000, 12
    dist = rng.uniform(-50, 90, size=(S, P, T, 2))
    dist[1, 7777, 3] = np.nan
    paths = [SimpleNamespace(t=np.arange(n) * pl.dt, x=rng.uniform(0, 40, n), y=rng.uniform(-5, 5, n),
                             yaw=np.zeros(n)) for n in (12, 5, 30)]
    got = pl.assess(paths, None, None, dist, r2=[[0.5, 0.0], [0.01, 0.0]])
    for j, p in enumerate(paths):
        ref = AO.assess_trajectory(p.t, p.x, p.y, p.yaw, pl.dt, dyn=dist, r2=[[0.5, 0.0], [0.01, 0.0]])
        assert _bits(got["dyn_min"][j]) == _bits(ref["dyn_min"])
        for name in ("dyn_at", "dyn_hits", "first_hit"):
            assert np.array_equal(got[name][j], ref[name]), (j, name)


# ---- 5. closed loop: the executed plan of every step, against the whole sample set ----------------------------------
@pytest.mark.parametrize("name", ["rollout_s01_best.npz", "rollout_s01_dist.npz"])
def test_closed_loop_assessment(name):
    """BatchedClosedLoop(assess=True) leaves every history bit for bit as assess=False leaves it, and its new columns
    are the restatement's, step by step, on the recorded plans against the recorded sample sets with their t = 0
    column -- the whole set even where planning used the representative sample."""
    import os
    from integrated_path_planning_b200.rollout import BatchedClosedLoop
    from tests.stub_sampler import batched_sampler
    from tests.test_gpu_rollout import HERE, _load, _sgan_knobs
    z = np.load(os.path.join(HERE, "golden", name))
    knobs, runs, _ = _load(name)
    sg = _sgan_knobs(z)
    tracks = np.stack([r["traj"] for r in runs])
    ego0 = np.stack([r["ego0"] for r in runs])
    outs, sims = [], []
    for assess in (False, True):
        seeds = [int(sg["gen_seed"]) + 1000 * i for i in range(len(runs))]
        sampler = batched_sampler(seeds, int(sg["num_samples"]), int(knobs["pred_len"]), float(sg["sigma"]))
        sim = BatchedClosedLoop(runs[0]["wx"], runs[0]["wy"], knobs, tracks, ego0, sampler=sampler, record=True,
                                assess=assess)
        sim.warmup()
        outs.append(sim.run())
        sims.append(sim)
    plain, assessed = outs
    assert set(assessed) == set(plain) | {"plan_min_distance", "plan_hit_fraction"}
    for key, v in plain.items():
        assert np.array_equal(v, assessed[key], equal_nan=v.dtype.kind == "f"), key
    for h0, h1 in zip(sims[0].history, sims[1].history):
        assert len(h0) == len(h1)
        for r0, r1 in zip(h0, h1):
            assert (r0["path"] is None) == (r1["path"] is None)
            if r0["path"] is not None:
                assert np.array_equal(_bits(r0["path"]), _bits(r1["path"]))
    own = sims[1].planner.engine.own_radii(2)
    n_checked = 0
    for i, h in enumerate(sims[1].history):
        for s, r in enumerate(h):
            got_min, got_frac = assessed["plan_min_distance"][i, s], assessed["plan_hit_fraction"][i, s]
            if r["path"] is None or r["path"].shape[1] < 2:            # no plan executed this step
                assert np.isnan(got_min) and np.isnan(got_frac), (i, s)
                continue
            if r["dist"] is None:
                continue
            dist = r["dist"]                                           # [S, P, T, 2], without the t = 0 column
            field = np.concatenate([np.broadcast_to(r["ped_pos"][None, :, None, :], (dist.shape[0],) + dist.shape[1:2] + (1, 2)),
                                    dist], axis=2)
            p = r["path"]
            ref = AO.assess_trajectory(p[0], p[9], p[10], p[11], sims[1].dt, static=sims[1].static_points, dyn=field,
                                       r2=own)
            assert _bits(got_min) == _bits(ref["dyn_min"]), (i, s)
            assert got_frac == ref["dyn_hits"][0] / dist.shape[0], (i, s)
            n_checked += 1
    assert n_checked > 20
