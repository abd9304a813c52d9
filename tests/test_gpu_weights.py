"""GPU: cost-weight sweeps (fot_select_weighted, fot_cost_terms) -- every query's winner under many weightings of the
six cost knobs from one sweep, and the five cost terms of every candidate.

The selection is held to three yardsticks: the winner of the same launch (for the handle's own weighting), a second
planner built with each weighting and run through the sweep, and the NumPy oracle built with that weighting."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import frenet_oracle as O
from tests import campaign, runners, scenarios

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
KEYS = ("k_j", "k_t", "k_d", "k_s_dot", "k_lat", "k_lon")


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


def _own(knobs):
    return np.array([float(knobs[k]) for k in KEYS])


def _weightings(knobs):
    """The handle's own, the reference's module defaults and the config defaults, each weight at 0 in turn and all six at
    0 (every cost ties at 0: the lowest feasible index wins), ratios 1e-3 .. 1e3, a NaN weight (no winner) and +inf
    (inf * 0 = NaN for some candidates)."""
    own = _own(knobs)
    w = [own, np.array([0.1, 0.1, 1.0, 1.0, 1.0, 1.0]), np.ones(6)]
    for i in range(6):
        z = own.copy()
        z[i] = 0.0
        w.append(z)
    w.append(np.zeros(6))
    w += [np.array([1e-3, 1e3, 1.0, 1e-3, 1e3, 1.0]), np.array([1e3, 1e-3, 1e3, 1.0, 1e-3, 1e3]),
          np.array([1.0, 1.0, 1e3, 1e-3, 1.0, 1.0])]
    nan, inf = own.copy(), own.copy()
    nan[2], inf[3] = np.nan, np.inf
    w += [nan, inf]
    return np.stack(w)


def _assert_own_weighting_is_the_winner(res, w=0):
    assert np.array_equal(res.w_idx[:, w], res.best_idx)
    assert np.array_equal(_bits(res.w_cost[:, w]), _bits(res.best_cost))
    assert np.array_equal(res.w_len[:, w], res.winner_len)
    for q in np.nonzero(res.best_idx >= 0)[0]:
        n = int(res.winner_len[q])
        assert np.array_equal(_bits(res.w_series[q, w, :, :n]), _bits(res.winner[q, :, :n])), q


def _assert_selection_equals_sweeps(knobs, wp, weights, run, planner_kw=None, n_min_found=1):
    """`run(planner, **extra)` plans the workload with plan_batch.  The selection under each weighting (shared, and per
    query with the list rotated by the query index) must equal a sweep of a planner built with that weighting: index,
    cost bits, stats and the winner series bits."""
    planner_kw = planner_kw or {}
    base = _planner(knobs, wp, **planner_kw)
    shared = run(base, cost_weights=weights)
    n_q, n_w = shared.w_idx.shape
    assert n_w == len(weights)
    _assert_own_weighting_is_the_winner(shared, 0)
    rot = np.array([np.roll(np.arange(n_w), q) for q in range(n_q)])         # query q's list: weights[rot[q]]
    per_q = run(base, cost_weights=weights[rot])
    n_found = 0
    for w in range(n_w):
        ref = run(_planner(dict(knobs, **dict(zip(KEYS, weights[w]))), wp, **planner_kw))
        assert np.array_equal(ref.stats, shared.stats), w
        found = ref.best_idx >= 0
        n_found += int(found.sum())
        pq_w = [np.nonzero(rot[q] == w)[0][0] for q in range(n_q)]             # column of weighting w in query q's list
        for res, col in ((shared, np.full(n_q, w)), (per_q, np.array(pq_w))):
            rows = np.arange(n_q)
            assert np.array_equal(res.w_idx[rows, col], ref.best_idx), (w, weights[w])
            assert np.array_equal(_bits(res.w_cost[rows, col]), _bits(ref.best_cost)), (w, weights[w])
            assert np.array_equal(res.w_len[rows, col][found], ref.winner_len[found]), w
            assert np.all(res.w_len[rows, col][~found] == 0), w
            for q in np.nonzero(found)[0]:
                n = int(ref.winner_len[q])
                assert np.array_equal(_bits(res.w_series[q, col[q], :, :n]), _bits(ref.winner[q, :, :n])), (w, q)
    nan_w = [w for w in range(n_w) if np.isnan(weights[w]).any()]
    assert all(np.all(shared.w_idx[:, w] == -1) and np.all(np.isposinf(shared.w_cost[:, w])) for w in nan_w)
    assert n_found >= n_min_found
    return shared


# ---- 1. the handle's own weighting reproduces the launch, on all three sweep kernels ------------------------------
@pytest.mark.parametrize("kernel", ["pairs", "items"])
def test_own_weighting_is_the_winner_config4(config4, kernel):
    frenet, dyn = config4
    pl = _planner()
    pl.engine
    w = _weightings(scenarios.S1_KNOBS)[:4]
    with runners.fot_env(FOT_SWEEP=kernel):
        res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0], cost_weights=w)
        assert int(pl.engine.lib.fot_last_sweep_kind(pl.engine._h)) == {"pairs": 4, "items": 1}[kernel]
    assert (res.best_idx >= 0).sum() > 100
    _assert_own_weighting_is_the_winner(res, 0)
    assert (res.w_idx[:, 1] != res.best_idx).sum() > 0                          # another weighting picks otherwise
    for q in np.nonzero(res.best_idx >= 0)[0][:32]:
        for e in res.under_weights(q):
            if e is not None:
                assert e["series"]["s"][0] == frenet[q, 0] and len(e["series"]["x"]) > 0


# ---- 2. the selection equals a sweep with those weights -------------------------------------------------------------
def test_selection_equals_sweeps_config4(config4):
    frenet, dyn = config4
    _assert_selection_equals_sweeps(scenarios.S1_KNOBS, scenarios.STRAIGHT_60, _weightings(scenarios.S1_KNOBS),
                                    lambda pl, **kw: pl.plan_batch(frenet[:128], 6.0, dynamic_obstacles=dyn[:128, 0], **kw),
                                    n_min_found=300)


def test_selection_equals_sweeps_near_limit_queries():
    """Campaign B: limits through the candidates' range (every category populated) and the stop-distance directive."""
    qs = [campaign.query_b(i) for i in range(campaign.N_B)]
    for path in campaign.PATH_NAMES:
        for road in (2.7, 1.1):
            ids = [i for i, q in enumerate(qs) if q["path"] == path and q["road"] == road]
            knobs = campaign.knobs_b(road)
            lim_pl = _planner(knobs, campaign.PATHS[path])
            limits = np.stack([lim_pl.resolve_limits(qs[i]["overrides"]) for i in ids])
            msd = np.array([np.nan if qs[i]["msd"] is None else qs[i]["msd"] for i in ids])
            fs = np.stack([qs[i]["fs"] for i in ids])
            target = np.array([qs[i]["target"] for i in ids])
            dyn = np.stack([qs[i]["dyn"] for i in ids])
            _assert_selection_equals_sweeps(
                knobs, campaign.PATHS[path], _weightings(knobs),
                lambda pl, **kw: pl.plan_batch(fs, target, dynamic_obstacles=dyn, limits=limits, max_stop_distance=msd, **kw))


@pytest.mark.parametrize("variant", [0, 1])
def test_selection_equals_sweeps_config3(variant):
    """66 563 candidates per query, distribution mode."""
    c = campaign.config3(variant)
    w = _weightings(c["knobs"])[[0, 1, 2, 4, 9, 10, 11, 13, 14]]
    res = _assert_selection_equals_sweeps(
        c["knobs"], c["waypoints"], w,
        lambda pl, **kw: pl.plan_batch(c["fs"][None], c["target"], distribution=c["dist"][None], **kw),
        n_min_found=0 if variant == 0 else 5)
    if variant == 0:
        assert np.all(res.w_idx == -1) and np.all(res.w_len == 0)


def test_selection_equals_sweeps_budgeted_distribution_with_footprint():
    rng = np.random.default_rng(5)
    n = 16
    knobs = dict(scenarios.S1_KNOBS, chance_epsilon=0.25)
    frenet = np.stack([rng.uniform(1, 10, n), rng.uniform(1, 7, n), rng.uniform(-1, 1, n),
                       rng.uniform(-1, 1, n), rng.normal(0, 0.2, n), rng.normal(0, 0.05, n)], axis=1)
    dists = []
    for i in range(n):
        r = np.random.default_rng(200 + i)
        base = scenarios.pedestrian_field(r, 14, x_range=(0.0, 20.0), y_range=(-5.0, 25.0))
        dists.append(scenarios.sample_distribution(r, base, 12, sigma=0.08))
    dist = np.stack(dists)
    _assert_selection_equals_sweeps(knobs, scenarios.arc_waypoints(), _weightings(knobs),
                                    lambda pl, **kw: pl.plan_batch(frenet, 6.0, distribution=dist, **kw),
                                    planner_kw=dict(footprint=runners.make_footprint((4.5, 2.0, 3))), n_min_found=20)


def test_selection_equals_sweeps_static_wall():
    rng = np.random.default_rng(3)
    n = 48
    k = scenarios.S1_KNOBS
    frenet = np.stack([rng.uniform(2, 30, n), rng.uniform(0, 8, n), rng.uniform(-1, 1, n),
                       rng.uniform(-1.5, 1.5, n), rng.normal(0, 0.3, n), rng.normal(0, 0.05, n)], axis=1)
    target = np.tile([6.0, 3.6, 0.0], n // 3)
    msd = np.where(target == 0.0, 5.0, np.nan)
    dyn = np.stack([scenarios.pedestrian_field(np.random.default_rng(50 + i), 30, x_range=(0.0, 70.0), y_range=(-8.0, 8.0))
                    for i in range(n)])
    wall = scenarios.wall(x=45.0, half=1.0, n=9)
    _assert_selection_equals_sweeps(k, scenarios.s_curve_waypoints(), _weightings(k),
                                    lambda pl, **kw: pl.plan_batch(frenet, target, dynamic_obstacles=dyn, static_obstacles=wall,
                                                                   max_stop_distance=msd, **kw), n_min_found=50)


def test_selection_equals_sweeps_long_time_grid():
    """129 samples per trajectory: fot_sweep_items runs, and the jerk sums take NumPy's split summation."""
    knobs = dict(scenarios.S1_KNOBS, dt=0.05, min_t=6.0, max_t=6.4, d_road_w=0.9, d_t_s=3.0)
    rng = np.random.default_rng(8)
    n = 16
    frenet = np.stack([rng.uniform(2, 10, n), rng.uniform(2, 6, n), np.zeros(n), rng.uniform(-1, 1, n),
                       np.zeros(n), np.zeros(n)], axis=1)
    dyn = np.stack([scenarios.pedestrian_field(rng, 5, n_steps=129, dt=0.05) for _ in range(n)])
    probe = _planner(knobs)
    assert probe.engine.n_t_max > 128
    _assert_selection_equals_sweeps(knobs, scenarios.STRAIGHT_60, _weightings(knobs),
                                    lambda pl, **kw: pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn, **kw), n_min_found=20)


# ---- 3. the oracle ---------------------------------------------------------------------------------------------
WALL_AHEAD = [scenarios.Query(f"wall_ahead_{x:.0f}", scenarios.S1_KNOBS, scenarios.STRAIGHT_60, (5.0, 0.0, 0.0, 5.0, 0.0),
                              6.0, static=scenarios.wall(x=x), overrides={"max_accel": 6.0}) for x in (16.0, 18.0)]


def _oracle_terms(cands, target_speed):
    """(Jp, Jd, Js, Jv, Jt) of every oracle candidate as generated (before truncation), with path_cost's expressions
    (oracle/frenet_oracle.py)."""
    return np.array([[np.sum(np.square(c.d_ddd)), (c.d[-1]) ** 2, np.sum(np.square(c.s_ddd)),
                      (target_speed - c.s_d[-1]) ** 2, c.t[-1]] for c in cands], dtype=np.float64)


def test_selection_and_terms_match_the_oracle():
    from integrated_path_planning_b200 import _lib
    from integrated_path_planning_b200.batch import DeviceBatch
    bad, n_exact, queries = [], 0, scenarios.standard_queries() + WALL_AHEAD
    for q in queries:
        weights = _weightings(q.knobs)[[0, 1, 4, 9, 10, 11]]
        winners = []
        pl = runners.cuda_planner(q)
        static = np.empty((0, 2)) if q.static is None else q.static
        paths = pl.plan_under_weights(runners._Ego(*q.ego), static, q.dyn, q.target_speed, q.overrides, q.dist,
                                      q.max_stop_distance, weights=weights)
        res_w = pl.last_result
        assert len(paths) == len(weights)
        for w, path in enumerate(paths):
            kn = O.Knobs(**dict(q.knobs, **dict(zip(KEYS, weights[w]))))
            fp = runners.make_footprint(q.footprint)
            if fp is not None:
                kn.footprint_offsets, kn.footprint_radius = fp.offsets, fp.radius
            orc = O.OraclePlanner(O.Spline2D(*q.waypoints), kn)
            orc.last_kappa = q.last_kappa
            ref = orc.plan(q.ego, static, q.dyn, q.target_speed, q.overrides, q.dist, q.max_stop_distance)
            got = int(res_w.w_idx[0, w])
            idx = np.arange(len(ref.categories))
            with np.errstate(invalid="ignore"):
                feas = idx[(ref.categories == O.CAT_OK) & (ref.costs < np.inf)]
            want = int(feas[np.lexsort((feas, ref.costs[feas]))][0]) if len(feas) else -1
            if got != want or (want >= 0 and _bits(res_w.w_cost[0, w]) != _bits(ref.costs[want])):
                bad.append((q.name, w, got, want))
                continue
            assert (path is None) == (want < 0), (q.name, w)
            if path is None:
                continue
            winners.append(want)
            cand = orc.last_candidates[want]
            for name in runners.SERIES:
                got_s, want_s = np.asarray(getattr(path, name), float), np.asarray(getattr(cand, name), float)
                assert got_s.shape == want_s.shape, (q.name, w, name)
                np.testing.assert_allclose(got_s, want_s, rtol=runners.RTOL, atol=runners.ATOL, err_msg=f"{q.name} {w} {name}")
        # the five cost terms of every candidate against the oracle's un-truncated candidates: within 1e-9 everywhere,
        # bit for bit for every candidate selected above (whose costs matched bit for bit)
        fs = np.asarray(runners.run_oracle(q).frenet_state, dtype=np.float64)
        db = DeviceBatch(pl, fs.reshape(1, 6), q.target_speed, None, _lib.FOT_DYN_NONE, cost_terms=True)
        db.launch()
        res = db.sweep_result()
        want_t = _oracle_terms(O.generate(O.Knobs(**q.knobs), fs, q.target_speed), q.target_speed)
        n_c = len(want_t)
        assert int(res.n_cand[0]) == n_c, q.name
        np.testing.assert_allclose(res.cost_terms[0, :n_c], want_t, rtol=runners.RTOL, atol=runners.ATOL, err_msg=q.name)
        assert np.array_equal(_bits(res.cost_terms[0, winners]), _bits(want_t[winners])), q.name
        n_exact += int(np.array_equal(_bits(res.cost_terms[0, :n_c]), _bits(want_t)))
        assert np.all(np.isnan(res.cost_terms[0, n_c:])), q.name
    assert not bad, bad
    assert n_exact >= len(queries) // 2, (n_exact, len(queries))   # most queries agree in every bit of every term


# ---- 4. the terms reproduce the table -------------------------------------------------------------------------------
def test_terms_reproduce_the_cost_table(config4):
    frenet, dyn = config4
    pl = _planner()
    res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[:, 0], top_k=1, cost_weights=_own(scenarios.S1_KNOBS)[None],
                        cost_terms=True, want_candidates=True)
    kj, kt, kd, ks, kla, klo = (float(x) for x in _own(scenarios.S1_KNOBS))
    n_checked = 0
    for q in range(0, len(frenet), 7):
        n_c = int(res.n_cand[q])
        assert np.all(np.isnan(res.cost_terms[q, n_c:])), q
        for i in np.nonzero(np.isfinite(res.cand_cost[q, :n_c]))[0]:
            jp, jd, js, jv, jt = (float(x) for x in res.cost_terms[q, i])
            lat = kj * jp + kt * jt + kd * jd                       # Python floats: one rounding per operation
            lon = kj * js + kt * jt + ks * jv
            assert _bits(kla * lat + klo * lon) == _bits(res.cand_cost[q, i]), (q, i)
            n_checked += 1
    assert n_checked > 10000


# ---- 5. the unweighted launch is unchanged ----------------------------------------------------------------------
def test_unweighted_launch_unchanged(config4):
    import torch
    from integrated_path_planning_b200 import _lib
    from integrated_path_planning_b200.batch import DeviceBatch
    frenet, dyn = config4
    pl = _planner()
    lib, h = pl.engine.lib, pl.engine._h
    plain = DeviceBatch(pl, frenet, 6.0, dyn, _lib.FOT_DYN_SINGLE)
    plain.launch()
    before = {k: v.cpu().numpy().copy() for k, v in plain.out.items()}
    feat = int(lib.fot_last_pair_features(h))
    assert feat == 0 and set(before) == {"best_idx", "best_cost", "stats", "winner_len", "winner"}
    weighted = DeviceBatch(pl, frenet, 6.0, dyn, _lib.FOT_DYN_SINGLE, cost_weights=_weightings(scenarios.S1_KNOBS),
                           cost_terms=True)
    weighted.launch()
    assert int(lib.fot_last_pair_features(h)) == 8                  # the instantiation with per-candidate outputs
    plain.launch()
    assert int(lib.fot_last_pair_features(h)) == feat
    torch.cuda.synchronize()
    after = {k: v.cpu().numpy() for k, v in plain.out.items()}
    w = {k: v.cpu().numpy() for k, v in weighted.out.items()}
    for key in ("best_idx", "stats", "winner_len"):
        assert np.array_equal(before[key], after[key]) and np.array_equal(before[key], w[key]), key
    assert np.array_equal(_bits(before["best_cost"]), _bits(after["best_cost"]))
    for q in np.nonzero(before["best_idx"] >= 0)[0]:
        n = int(before["winner_len"][q])
        assert np.array_equal(_bits(before["winner"][q, :, :n]), _bits(after["winner"][q, :, :n])), q
    host = {k: np.zeros(v.shape, dtype=v.dtype) for k, v in before.items()}
    with pytest.raises(ValueError):
        weighted.launch_to_host(host)


# ---- 6. plan_under_weights in lock-step with plan() ------------------------------------------------------------
def test_plan_under_weights_lock_step_with_plan():
    from integrated_path_planning_b200 import CubicSpline2D, FrenetPlanner
    store = runners.load_golden("closed_loop_s01.npz")
    wp = (store["waypoints_x"], store["waypoints_y"])
    one = FrenetPlanner(CubicSpline2D(*wp), **scenarios.S1_KNOBS)
    wtd = FrenetPlanner(CubicSpline2D(*wp), **scenarios.S1_KNOBS)
    weights = [{"k_d": 5.0}, {}, {"k_j": 0.1, "k_lon": 3.0}]           # entry 1 is the planner's own weighting
    n_found = n_differs = 0
    for j in range(len(store["kept"])):
        g = runners.golden_case(store, f"c{j}")
        for pl in (one, wtd):
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
        paths = wtd.plan_under_weights(*args, weights=weights)
        assert len(paths) == 3
        assert one.last_check_stats == wtd.last_check_stats, j
        assert one._last_kappa == wtd._last_kappa, j
        assert getattr(one.converter, "_prev_s", None) == getattr(wtd.converter, "_prev_s", None), j
        assert (path is None) == (paths[1] is None), j
        if path is None:
            continue
        n_found += 1
        n_differs += int(paths[0] is not None and float(paths[0].cost) != float(path.cost))
        assert _bits(paths[1].cost) == _bits(path.cost), j
        for name in runners.SERIES:
            assert np.array_equal(_bits(getattr(paths[1], name)), _bits(getattr(path, name))), (j, name)
            assert type(getattr(paths[1], name)) is type(getattr(path, name)), (j, name)
    assert n_found > 0 and n_differs > 0


# ---- 7. roll-out ------------------------------------------------------------------------------------------------
def _load_rollout(name):
    z = np.load(os.path.join(HERE, "golden", name))
    knobs = {k[5:]: float(z[k]) for k in z.files if k.startswith("knob/")}
    runs = [{key: z[f"v{i}/{key}"] for key in ("traj", "ego0", "wx", "wy")} for i in range(int(z["n_variants"]))]
    sg = {k[5:]: float(z[k]) for k in z.files if k.startswith("sgan/")}
    return knobs, runs, sg


@pytest.mark.parametrize("name", ["rollout_s01.npz", "rollout_s01_dist.npz"])
def test_rollout_groups_equal_separate_rollouts(name):
    """The four variants under three weightings each, 12 simulations in one BatchedClosedLoop(cost_weights=...), equal
    three separate roll-outs built with those knobs; the group with the base knobs equals a run without weights."""
    from integrated_path_planning_b200.rollout import BatchedClosedLoop
    knobs, runs, sg = _load_rollout(name)
    base = _own(knobs)
    groups = [base, base * np.array([1.0, 1.0, 5.0, 0.2, 1.0, 1.0]), base * np.array([0.1, 1.0, 1.0, 1.0, 1.0, 3.0])]
    n_v = len(runs)

    def sampler(n):
        if not sg:
            return None
        from tests.stub_sampler import batched_sampler
        seeds = [int(sg["gen_seed"]) + 1000 * (i % n_v) for i in range(n)]
        return batched_sampler(seeds, int(sg["num_samples"]), int(knobs["pred_len"]), float(sg["sigma"]))

    def drive(kn, reps, weights=None):
        tracks = np.concatenate([np.stack([r["traj"] for r in runs])] * reps)
        ego0 = np.concatenate([np.stack([r["ego0"] for r in runs])] * reps)
        sim = BatchedClosedLoop(runs[0]["wx"], runs[0]["wy"], kn, tracks, ego0, sampler=sampler(n_v * reps),
                                cost_weights=weights)
        sim.warmup()
        return sim.run()

    together = drive(knobs, 3, np.repeat(np.stack(groups), n_v, axis=0))
    n_steps = together["ego"].shape[1]
    differ = 0
    for g, w in enumerate(groups):
        alone = drive(dict(knobs, **dict(zip(KEYS, w))), 1)
        rows = slice(g * n_v, (g + 1) * n_v)
        assert alone["ego"].shape[1] == n_steps
        for key in ("ego", "fsm", "found", "calls", "reason", "steps"):
            np.testing.assert_array_equal(together[key][rows], alone[key], err_msg=f"group {g} {key}")
        if g > 0:
            differ += int(not np.array_equal(together["ego"][rows], together["ego"][:n_v]))
    assert differ > 0                                                 # the weightings do change the roll-outs


# ---- 8. argument errors -----------------------------------------------------------------------------------------
def test_rejects_bad_arguments(config4):
    from integrated_path_planning_b200 import _lib
    from integrated_path_planning_b200.batch import DeviceBatch
    frenet, dyn = config4
    pl = _planner()
    w = _weightings(scenarios.S1_KNOBS)[:3]
    db = DeviceBatch(pl, frenet[:16], 6.0, dyn[:16], _lib.FOT_DYN_SINGLE, cost_weights=w, cost_terms=True)
    db.launch()
    eng = pl.engine
    good_len = db.out["w_len"].cpu().numpy().copy()

    def call(batch=None, weighted=None, stride=None, cat=None):
        eng.select_weighted_device(batch or db.batch, db.result.cand_cat if cat is None else cat,
                                   db.stride if stride is None else stride, weighted or db.weighted)

    def weighted(**kw):
        x = _lib.FotWeighted.from_buffer_copy(db.weighted)
        for key, v in kw.items():
            setattr(x, key, v)
        return x

    empty = _lib.FotBatch.from_buffer_copy(db.batch)
    empty.n_q = 0
    no_target = _lib.FotBatch.from_buffer_copy(db.batch)
    no_target.target_speed = None
    bad_calls = [dict(weighted=weighted(n_w=0)), dict(weighted=weighted(n_w=_lib.FOT_MAX_WEIGHT_SETS + 1)),
                 dict(weighted=weighted(weights=None)), dict(weighted=weighted(idx=None)), dict(weighted=weighted(cost=None)),
                 dict(weighted=weighted(len=None)), dict(weighted=weighted(per_query=2)), dict(stride=db.stride - 1),
                 dict(batch=empty), dict(batch=no_target), dict(cat=0)]
    for kw in bad_calls:
        with pytest.raises(_lib.FotError):
            call(**kw)
    for kw in (dict(stride=db.stride - 1), dict(batch=empty), dict(terms=0)):
        with pytest.raises(_lib.FotError):
            eng.cost_terms_device(kw.get("batch", db.batch), kw.get("stride", db.stride),
                                  kw.get("terms", db.out["cost_terms"].data_ptr()))
    # lengths without series are allowed; they equal the lengths that come with the series
    db.out["w_len"].fill_(-5)
    call(weighted=weighted(series=None))
    assert np.array_equal(db.out["w_len"].cpu().numpy(), good_len)
    assert int(C.sizeof(_lib.FotWeighted)) == 48
    # the Python layers
    for bad in (np.ones((0, 6)), np.ones((_lib.FOT_MAX_WEIGHT_SETS + 1, 6)), np.ones((3, 5)), np.ones((15, 3, 6)),
                np.ones(6)):
        with pytest.raises(ValueError):
            DeviceBatch(pl, frenet[:16], 6.0, dyn[:16], _lib.FOT_DYN_SINGLE, cost_weights=bad)
    with pytest.raises(ValueError):
        pl.plan_batch(frenet[:16], 6.0, dynamic_obstacles=dyn[:16, 0], cost_weights=np.ones((4, 7)))
    ego = runners._Ego(5.0, 0.0, 0.0, 5.0, 0.0)
    for bad in (np.ones((0, 6)), [{"k_x": 1.0}], np.ones((2, 5))):
        with pytest.raises(ValueError):
            pl.plan_under_weights(ego, np.empty((0, 2)), weights=bad)
    host = {k: np.zeros(v.shape, dtype=v.cpu().numpy().dtype) for k, v in db.out.items()}
    with pytest.raises(ValueError):
        db.launch_to_host(host)
