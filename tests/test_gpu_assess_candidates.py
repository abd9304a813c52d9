"""GPU: candidate assessment (fot_assess_candidates) against the NumPy restatement (tests/assess_oracle.py) on the
oracle's candidates, against fot_assess_trajectories on the ranked series, against the sweep's own categories, and on
the edge and size cases."""
import numpy as np
import pytest

from oracle import frenet_oracle as O
from tests import assess_oracle as AO
from tests import campaign, runners, scenarios

pytestmark = pytest.mark.gpu

NAMES = ("dyn_min", "dyn_at", "static_min", "static_at", "dyn_hits", "first_hit", "static_hit")


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _planner(wp, knobs, footprint=None):
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    return BatchFrenetPlanner(CubicSpline2D(*wp), footprint=runners.make_footprint(footprint), **knobs)


def _check_rows(cands, got, dt, static, field, r2, offsets, exact):
    """Row i of `got` (one query's candidate table) against the restatement on oracle candidate i (generation order)."""
    assert len(got["keep"]) == len(cands)
    assert got["keep"].tolist() == [c.keep for c in cands]
    bad = []
    for i, c in enumerate(cands):
        if c.keep == 0:
            ok = got["dyn_min"][i] == np.inf and got["static_min"][i] == np.inf and np.all(got["dyn_at"][i] == -1)
            ok &= np.all(got["dyn_hits"][i] == 0) and np.all(got["first_hit"][i] == -1) and np.all(got["static_hit"][i] == 0)
            if not ok:
                bad.append((i, "blank"))
            continue
        ref = AO.assess_trajectory(c.t, c.x, c.y, c.yaw, dt, static=static, dyn=field, r2=r2, offsets=offsets)
        if exact:
            ok = _bits(got["dyn_min"][i]) == _bits(ref["dyn_min"]) and _bits(got["static_min"][i]) == _bits(ref["static_min"])
        else:
            ok = all(np.isclose(got[k][i], ref[k], rtol=1e-12, atol=0) or got[k][i] == ref[k] for k in ("dyn_min", "static_min"))
        for name in ("dyn_at", "static_at", "dyn_hits", "first_hit", "static_hit"):
            ok &= np.array_equal(got[name][i], ref[name])
        if not ok:
            bad.append((i, {k: got[k][i] for k in NAMES}, ref))
    assert not bad, (f"{len(bad)} of {len(cands)} differ", bad[0])


def _free(a, allowed):
    return (a["static_hit"][..., 0] == 0) & (a["dyn_hits"][..., 0] <= allowed)


def _check_categories(cat, ca, n_cand, allowed):
    """Under the handle's own pair: OK and STOP candidates are free, COLL candidates are not."""
    cols = np.arange(cat.shape[1])[None, :] < np.asarray(n_cand)[:, None]
    free = _free(ca, allowed)
    ok_or_stop = cols & ((cat == O.CAT_OK) | (cat == O.CAT_STOP))
    coll = cols & (cat == O.CAT_COLL)
    assert ok_or_stop.any() or coll.any()
    assert np.all(free[ok_or_stop]), np.argwhere(ok_or_stop & ~free)[:5]
    assert not np.any(free[coll]), np.argwhere(coll & free)[:5]
    # columns past the candidates are blank
    assert np.all(ca["keep"][~cols] == 0) and np.all(np.isposinf(ca["dyn_min"][~cols])) and np.all(ca["first_hit"][~cols] == -1)


# ---- 1. against the restatement on the oracle's candidates ----------------------------------------------------------
@pytest.mark.parametrize("q", scenarios.standard_queries(), ids=lambda q: q.name)
def test_standard_queries_against_oracle(q):
    opl = runners.oracle_planner(q)
    static = np.empty((0, 2)) if q.static is None else q.static
    opl.plan(q.ego, static, q.dyn, q.target_speed, q.overrides, q.dist, q.max_stop_distance)
    cands = opl.last_candidates
    pl = runners.cuda_planner(q)
    dist_mode = q.dist is not None
    own = pl.engine.own_radii(2 if dist_mode else 1)
    r2 = np.concatenate([own, [[own[0, 0] * 4.0, own[0, 1] * 0.25], [0.0, 0.0], [1.0, 9.0]]])
    got = pl.candidate_assessment(runners._Ego(*q.ego), static, q.dyn, q.target_speed, q.overrides, q.dist,
                                  q.max_stop_distance, r2=r2)
    field = q.dist if dist_mode else (None if q.dyn is None else q.dyn[None])
    # bit for bit with the single circle on the straight path; on a curved one the spline's positions carry the 1-ulp
    # deviations of DESIGN.md section 7, and with footprint circles CUDA's cos / sin
    exact = opl.k.footprint_offsets is None and q.waypoints == scenarios.STRAIGHT_60
    _check_rows(cands, got, opl.k.dt, static, field, r2, opl.k.footprint_offsets, exact=exact)
    assert got["cand_cat"].astype(np.int8).tolist() == [c.category for c in cands]
    # side effects are plan()'s
    ref_stats = runners.run_cuda(q)[0].last_check_stats
    assert pl.last_check_stats == ref_stats


@pytest.mark.parametrize("i", range(0, 42, 3))
def test_campaign_b_against_oracle(i):
    b = campaign.query_b(i)
    kn = O.Knobs(**campaign.knobs_b(b["road"]))
    opl = O.OraclePlanner(O.Spline2D(*campaign.PATHS[b["path"]]), kn)
    opl.plan_frenet(b["fs"], None, b["dyn"], b["target"], b["overrides"], None, b["msd"])
    pl = _planner(campaign.PATHS[b["path"]], campaign.knobs_b(b["road"]))
    res = pl.plan_batch(b["fs"][None], b["target"], dynamic_obstacles=b["dyn"][None], constraint_overrides=b["overrides"],
                        max_stop_distance=b["msd"], want_candidates=True, assess_candidates=True)
    got = res.candidate_assessment(0)
    _check_rows(opl.last_candidates, got, kn.dt, None, b["dyn"][None], pl.engine.own_radii(1), None, exact=True)
    assert got["cand_cat"].astype(np.int8).tolist() == [c.category for c in opl.last_candidates]


# ---- 2. against fot_assess_trajectories on the ranked series --------------------------------------------------------
@pytest.fixture(scope="module")
def config4():
    import bench
    _, frenet, dyn = bench.make_queries(3000, 512)
    return frenet, dyn


@pytest.mark.parametrize("footprint", [None, (4.5, 2.0, 3)])
def test_ranked_columns_equal_trajectory_assessment(config4, footprint):
    frenet, dyn = config4
    pl = _planner(scenarios.STRAIGHT_60, scenarios.S1_KNOBS, footprint)
    own = pl.engine.own_radii(1)
    r2 = np.concatenate([own, [[9.0, 9.0], [0.25, 0.0]]])
    res = pl.plan_batch(frenet[:256], 6.0, dynamic_obstacles=dyn[:256, 0], top_k=32, assess=True, assess_candidates=True,
                        assess_r2=r2)
    has = res.rank_idx >= 0
    assert has.sum() > 256
    qs, rs = np.nonzero(has)
    idx = res.rank_idx[qs, rs]
    for name in NAMES:
        a, c = res.assessed[name][qs, rs], res.cand_assessed[name][qs, idx]
        diff = (_bits(a) != _bits(c)) if a.dtype == np.float64 else (a != c).reshape(len(a), -1).any(axis=1)
        j = np.flatnonzero(diff)
        assert j.size == 0, (name, j.size, len(a), qs[j[:3]], rs[j[:3]], idx[j[:3]], a[j[:3]], c[j[:3]])
    assert np.array_equal(res.cand_assessed["keep"][qs, idx], res.rank_len[qs, rs])


# ---- 3. against the sweep's categories -------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", ["pairs", "items"])
def test_categories_config4(config4, kernel):
    frenet, dyn = config4
    pl = _planner(scenarios.STRAIGHT_60, scenarios.S1_KNOBS)
    pl.engine
    with runners.fot_env(FOT_SWEEP=kernel):
        res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0], want_candidates=True, assess_candidates=True)
    _check_categories(res.cand_cat, res.cand_assessed, res.n_cand, 0)


def test_categories_campaign_b():
    n_coll = 0
    for i in range(42):
        b = campaign.query_b(i)
        pl = _planner(campaign.PATHS[b["path"]], campaign.knobs_b(b["road"]))
        res = pl.plan_batch(b["fs"][None], b["target"], dynamic_obstacles=b["dyn"][None],
                            constraint_overrides=b["overrides"], max_stop_distance=b["msd"], want_candidates=True,
                            assess_candidates=True)
        a = res.candidate_assessment(0)
        free = _free(a, 0)
        cat = a["cand_cat"]
        assert np.all(free[(cat == O.CAT_OK) | (cat == O.CAT_STOP)]) and not np.any(free[cat == O.CAT_COLL]), i
        n_coll += int((cat == O.CAT_COLL).sum())
    assert n_coll > 0


def test_categories_budgeted_distribution_with_footprint():
    rng = np.random.default_rng(41)
    k = dict(scenarios.S1_KNOBS, chance_epsilon=0.2)
    pl = _planner(scenarios.s_curve_waypoints(), k, (4.5, 2.0, 3))
    n_q, S = 64, 10
    frenet = np.zeros((n_q, 6))
    frenet[:, 0], frenet[:, 1], frenet[:, 3] = rng.uniform(3, 20, n_q), rng.uniform(1, 6, n_q), rng.uniform(-1, 1, n_q)
    base = np.stack([scenarios.pedestrian_field(rng, 14, x_range=(5.0, 45.0), y_range=(-4.0, 6.0)) for _ in range(n_q)])
    dist = np.stack([scenarios.sample_distribution(rng, base[q], S, sigma=0.2) for q in range(n_q)])
    res = pl.plan_batch(frenet, 6.0, distribution=dist, want_candidates=True, assess_candidates=True)
    _check_categories(res.cand_cat, res.cand_assessed, res.n_cand, int(np.floor(0.2 * S)))
    budget = res.cand_assessed["dyn_hits"][..., 0]
    assert np.any((budget > 0) & (budget <= 2) & (res.cand_cat == O.CAT_OK))     # the budget is used


@pytest.mark.parametrize("name", ["single", "footprint", "distribution"])
def test_categories_collision_boundary_scenes(name):
    from tests import test_gpu_collision_boundary as CB
    names = [k for k in CB.SETUPS if (name == "footprint") == bool(CB.SETUPS[k].footprint) and
             (name == "distribution") == bool(CB.SETUPS[k].dist_s)]
    assert names
    for key in names:
        s = CB.SETUPS[key]
        frenet, dyn, stat = CB.batch(key)
        pl = _planner(s.wp, s.knobs, s.footprint)
        kw = dict(distribution=dyn) if s.dist_s else dict(dynamic_obstacles=dyn[:, 0])
        res = pl.plan_batch(frenet, s.target_speed, static_obstacles=stat, want_candidates=True, assess_candidates=True,
                            **kw)
        allowed = int(np.floor(pl.chance_epsilon * dyn.shape[1])) if s.dist_s else 0
        cols = np.arange(res.cand_cat.shape[1])[None, :] < res.n_cand[:, None]
        free = _free(res.cand_assessed, allowed)
        cat = res.cand_cat
        assert np.all(free[cols & ((cat == O.CAT_OK) | (cat == O.CAT_STOP))]), key
        assert not np.any(free[cols & (cat == O.CAT_COLL)]), key


@pytest.mark.parametrize("kernel", ["pairs", "items"])
def test_categories_config3_shape(kernel):
    rng = np.random.default_rng(33)
    knobs = dict(scenarios.S1_KNOBS, d_road_w=0.1, max_road_width=3.2, min_t=1.9, max_t=5.0, d_t_s=0.2)
    wp = (np.linspace(0.0, 80.0, 9).tolist(), [0.0] * 9)
    base = scenarios.pedestrian_field(rng, 200, x_range=(5.0, 65.0), vel_clip=2.5)
    dist = scenarios.sample_distribution(rng, base, 20)
    pl = _planner(wp, knobs)
    pl.engine
    fs = np.array([[5.0, 5.0, 0.0, 0.0, 0.0, 0.0]])
    with runners.fot_env(FOT_SWEEP=kernel):
        res = pl.plan_batch(fs, 6.2, distribution=dist[None], want_candidates=True, assess_candidates=True)
    assert int(res.n_cand[0]) == 66563
    _check_categories(res.cand_cat, res.cand_assessed, res.n_cand, 0)


# ---- 4. edge and shape cases -----------------------------------------------------------------------------------------
def test_nan_at_sample_one_and_singular_candidates_keep_zero():
    """A query whose s leaves the path at sample 1 (every grid candidate kept 0), and the tight arc, whose singular
    candidates the reference empties (fp.py:826-833): keep equals the oracle's, and those columns are blank."""
    k = scenarios.S1_KNOBS
    pl = _planner(scenarios.STRAIGHT_60, k)
    frenet = np.array([[59.5, 8.0, 0.0, 0.2, 0.0, 0.0], [30.0, 5.0, 0.0, 0.0, 0.0, 0.0]])
    dyn = np.stack([scenarios.pedestrian_field(np.random.default_rng(q), 5) for q in range(2)])
    res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn, assess_candidates=True)
    opl = O.OraclePlanner(O.Spline2D(*scenarios.STRAIGHT_60), O.Knobs(**k))
    for q in range(2):
        opl.plan_frenet(tuple(frenet[q]), None, dyn[q], 6.0)
        a = res.candidate_assessment(q)
        assert a["keep"].tolist() == [c.keep for c in opl.last_candidates], q
    first = res.candidate_assessment(0)
    assert np.all(first["keep"] == 0) and np.all(np.isposinf(first["dyn_min"])) and np.all(first["dyn_at"] == -1)
    tight = [q for q in scenarios.standard_queries() if q.name == "tight_arc_singularity"][0]
    opl = runners.oracle_planner(tight)
    opl.plan(tight.ego, np.empty((0, 2)), None, tight.target_speed)
    n_sing = sum(c.keep == 0 and c.category == O.CAT_DROP for c in opl.last_candidates)
    got = runners.cuda_planner(tight).candidate_assessment(runners._Ego(*tight.ego), None, None, tight.target_speed)
    assert got["keep"].tolist() == [c.keep for c in opl.last_candidates] and n_sing > 0


def test_bad_route_ids_give_blank_columns(config4):
    frenet, dyn = config4
    from integrated_path_planning_b200 import DeviceBatch
    pl = _planner(scenarios.STRAIGHT_60, scenarios.S1_KNOBS)
    from integrated_path_planning_b200 import CubicSpline2D
    pl.add_route(CubicSpline2D(*scenarios.s_curve_waypoints()))
    route = np.arange(16) % 2
    db = DeviceBatch(pl, frenet[:16], 6.0, dyn[:16], 1, route=route, assess_candidates=True)
    db.t["route"][3] = 7
    db.t["route"][8] = -1
    db.launch()
    res = db.sweep_result()
    ref = pl.plan_batch(frenet[:16], 6.0, dynamic_obstacles=dyn[:16, 0], route=route, assess_candidates=True)
    for q in range(16):
        a, r = res.cand_assessed, ref.cand_assessed
        if q in (3, 8):
            assert np.all(a["keep"][q] == 0) and np.all(np.isposinf(a["dyn_min"][q])) and np.all(a["dyn_at"][q] == -1)
            assert np.all(a["dyn_hits"][q] == 0) and np.all(a["first_hit"][q] == -1), q
            assert res.best_idx[q] == -1
        else:
            assert np.array_equal(_bits(a["dyn_min"][q]), _bits(r["dyn_min"][q])), q
            assert np.array_equal(a["dyn_at"][q], r["dyn_at"][q]) and np.array_equal(a["keep"][q], r["keep"][q]), q


def test_per_query_static_points_against_oracle():
    rng = np.random.default_rng(8)
    k = scenarios.S1_KNOBS
    pl = _planner(scenarios.STRAIGHT_60, k)
    n_q = 4
    frenet = np.zeros((n_q, 6))
    frenet[:, 0], frenet[:, 1], frenet[:, 3] = rng.uniform(3, 10, n_q), rng.uniform(2, 6, n_q), rng.uniform(-1, 1, n_q)
    dyn = np.stack([scenarios.pedestrian_field(rng, 8) for _ in range(n_q)])
    dyn[1, 2, 7] = (np.nan, 1.0)
    static = np.stack([scenarios.wall(x=20.0 + 4 * q, half=2.0, n=9) for q in range(n_q)])
    r2 = np.array([[1.44, 1.44], [9.0, 25.0]])
    res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn, static_obstacles=static, assess_candidates=True, assess_r2=r2)
    opl = O.OraclePlanner(O.Spline2D(*scenarios.STRAIGHT_60), O.Knobs(**k))
    for q in range(n_q):
        opl.plan_frenet(tuple(frenet[q]), static[q], dyn[q], 6.0)
        _check_rows(opl.last_candidates, res.candidate_assessment(q), k["dt"], static[q], dyn[q][None], r2, None, True)


def test_another_field_the_sample_set_with_its_t0_column():
    rng = np.random.default_rng(21)
    k = dict(scenarios.S1_KNOBS, chance_epsilon=0.2)
    pl = _planner(scenarios.STRAIGHT_60, k)
    n_q, S, P = 6, 20, 10
    frenet = np.zeros((n_q, 6))
    frenet[:, 0], frenet[:, 1], frenet[:, 3] = rng.uniform(3, 10, n_q), rng.uniform(2, 6, n_q), rng.uniform(-1, 1, n_q)
    base = np.stack([scenarios.pedestrian_field(rng, P, x_range=(5.0, 30.0), y_range=(-3.0, 3.0)) for _ in range(n_q)])
    dist = np.stack([scenarios.sample_distribution(rng, base[q], S, sigma=0.15) for q in range(n_q)])
    now = np.broadcast_to(base[:, None, :, :1], (n_q, S, P, 1, 2))
    field = np.ascontiguousarray(np.concatenate([now, dist[:, :, :, 1:]], axis=3))
    res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dist[:, 0], assess_candidates=True, assess_obstacles=field)
    opl = O.OraclePlanner(O.Spline2D(*scenarios.STRAIGHT_60), O.Knobs(**k))
    n_hit = 0
    for q in range(n_q):
        opl.plan_frenet(tuple(frenet[q]), None, dist[q, 0], 6.0)
        got = res.candidate_assessment(q)
        _check_rows(opl.last_candidates, got, k["dt"], None, field[q], pl.engine.own_radii(2), None, True)
        n_hit += int((got["dyn_hits"][:, 0] > 1).sum())
    assert n_hit > 0


def _sampled_rows(res, q, cands, every):
    """Every `every`-th kept candidate of query q: (oracle candidates, the matching rows of the table)."""
    got = res.candidate_assessment(q)
    assert got["keep"].tolist() == [c.keep for c in cands]
    pick = [i for i in range(len(cands)) if cands[i].keep > 0][::every]
    return [cands[i] for i in pick], {k: v[pick] for k, v in got.items()}


def test_long_grid_eight_circles_and_several_passes():
    """A 320-sample time grid with 8 footprint circles, against a field of 40 samples (two passes of samples)."""
    from tests.test_gpu_long_grids import LONG_STRAIGHT
    rng = np.random.default_rng(320)
    knobs = dict(scenarios.S1_KNOBS, dt=0.05, min_t=15.6, max_t=15.95, d_road_w=0.9, d_t_s=3.0)
    pl = _planner(LONG_STRAIGHT, knobs, (4.5, 2.0, 8))
    assert pl.engine.n_t_max == 320
    frenet = np.array([[5.0, 4.0, 0.0, 0.3, 0.0, 0.0], [8.0, 5.5, 0.1, -0.5, 0.1, 0.0]])
    field = np.stack([scenarios.sample_distribution(rng, scenarios.pedestrian_field(
        rng, 8, n_steps=330, dt=0.05, x_range=(10.0, 90.0), y_range=(-4.0, 4.0)), 40, sigma=0.1) for _ in range(2)])
    field[0, 3, 5, 17] = np.nan
    static = np.stack([rng.uniform(0.0, 90.0, size=5), rng.uniform(-4.0, 4.0, size=5)], axis=1)
    r2 = np.array([[1.0, 1.0], [0.04, 9.0], [16.0, 0.0]])
    res = pl.plan_batch(frenet, 6.0, static_obstacles=static, assess_candidates=True, assess_obstacles=field, assess_r2=r2)
    opl = O.OraclePlanner(O.Spline2D(*LONG_STRAIGHT), O.Knobs(**knobs))
    offsets = runners.make_footprint((4.5, 2.0, 8)).offsets
    n_hit = 0
    for q in range(2):
        opl.plan_frenet(tuple(frenet[q]), static, None, 6.0)
        cands, got = _sampled_rows(res, q, opl.last_candidates, 9)
        _check_rows(cands, got, knobs["dt"], static, field[q], r2, offsets, exact=False)
        n_hit += int((got["dyn_hits"][:, 2] > 32).sum())
    assert n_hit > 0                                                   # hits counted in both passes


def test_field_above_32768_trajectories():
    rng = np.random.default_rng(6)
    k = scenarios.S1_KNOBS
    pl = _planner(scenarios.STRAIGHT_60, k)
    S, P, T = 3, 11000, 12
    field = rng.uniform(-10.0, 70.0, size=(1, S, P, T, 2))
    field[0, 1, 7777, 3] = np.nan
    frenet = np.array([[5.0, 4.0, 0.0, 0.3, 0.0, 0.0]])
    r2 = np.array([[0.5, 0.0], [0.01, 0.0]])
    res = pl.plan_batch(frenet, 6.0, assess_candidates=True, assess_obstacles=field, assess_r2=r2)
    opl = O.OraclePlanner(O.Spline2D(*scenarios.STRAIGHT_60), O.Knobs(**k))
    opl.plan_frenet(tuple(frenet[0]), None, None, 6.0)
    cands, got = _sampled_rows(res, 0, opl.last_candidates, 60)
    _check_rows(cands, got, k["dt"], None, field[0], r2, None, exact=True)


def test_routed_batch_matches_per_route_planners(config4):
    frenet, dyn = config4
    paths = [scenarios.STRAIGHT_60, scenarios.s_curve_waypoints()]
    pl = _planner(paths[0], scenarios.S1_KNOBS)
    from integrated_path_planning_b200 import CubicSpline2D
    pl.add_route(CubicSpline2D(*paths[1]))
    route = np.arange(48) % 2
    res = pl.plan_batch(frenet[:48], 6.0, dynamic_obstacles=dyn[:48, 0], route=route, assess_candidates=True)
    for rid, wp in enumerate(paths):
        sel = np.nonzero(route == rid)[0]
        ref = _planner(wp, scenarios.S1_KNOBS).plan_batch(frenet[sel], 6.0, dynamic_obstacles=dyn[sel, 0],
                                                          assess_candidates=True)
        for name in ("dyn_min", "static_min"):
            assert np.array_equal(_bits(res.cand_assessed[name][sel]), _bits(ref.cand_assessed[name])), (rid, name)
        for name in ("dyn_at", "static_at", "dyn_hits", "first_hit", "static_hit", "keep"):
            assert np.array_equal(res.cand_assessed[name][sel], ref.cand_assessed[name]), (rid, name)


def test_launch_to_host_refuses_and_from_ego_blanks_failed_rows(config4):
    frenet, dyn = config4
    from integrated_path_planning_b200 import DeviceBatch
    pl = _planner(scenarios.STRAIGHT_60, scenarios.S1_KNOBS)
    db = DeviceBatch(pl, frenet[:4], 6.0, dyn[:4], 1, assess_candidates=True)
    with pytest.raises(ValueError, match="candidate assessments"):
        db.launch_to_host({})
    ego = np.array([[5.0, 0.0, 0.0, 5.0, 0.0], [np.nan, 0.0, 0.0, 5.0, 0.0], [12.0, 0.3, 0.0, 4.0, 0.0]])
    res, ok = pl.plan_batch_from_ego(ego, 6.0, dynamic_obstacles=dyn[:3, 0], assess_candidates=True)
    a = res.cand_assessed
    assert ok[0] and ok[2] and np.any(a["keep"][0] > 0) and np.any(a["keep"][2] > 0)
    for q in np.flatnonzero(~ok):                                       # plan() would return None: blank rows
        assert np.all(a["keep"][q] == 0) and np.all(np.isposinf(a["dyn_min"][q])) and np.all(a["first_hit"][q] == -1)


# ---- 5. existing outputs unchanged -----------------------------------------------------------------------------------
def test_other_outputs_unchanged(config4):
    frenet, dyn = config4
    pl = _planner(scenarios.STRAIGHT_60, scenarios.S1_KNOBS)
    w = np.array([[1.0, 1.0, 1.0, 1.0, 1.0, 1.0], [0.5, 2.0, 1.0, 3.0, 1.0, 0.7]])
    kw = dict(dynamic_obstacles=dyn[:128, 0], top_k=4, cost_weights=w, assess=True, cost_terms=True)
    a = pl.plan_batch(frenet[:128], 6.0, **kw)
    b = pl.plan_batch(frenet[:128], 6.0, assess_candidates=True, **kw)
    assert b.cand_assessed is not None and a.cand_assessed is None
    for name in ("best_idx", "best_cost", "stats", "winner_len", "rank_idx", "rank_cost", "rank_len", "w_idx", "w_cost",
                 "w_len", "cost_terms"):
        x, y = getattr(a, name), getattr(b, name)
        assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), name
    for q in np.nonzero(a.best_idx >= 0)[0]:
        n = int(a.winner_len[q])
        assert np.array_equal(_bits(a.winner[q, :, :n]), _bits(b.winner[q, :, :n])), q
    for q, r in zip(*np.nonzero(a.rank_idx >= 0)):
        n = int(a.rank_len[q, r])
        assert np.array_equal(_bits(a.rank_series[q, r, :, :n]), _bits(b.rank_series[q, r, :, :n])), (q, r)
    for name in NAMES:
        assert np.array_equal(a.assessed[name], b.assessed[name]), name
