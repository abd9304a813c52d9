"""GPU: the differential campaign against answers recorded from the UNMODIFIED reference
(tests/golden/make_golden_campaign.py; inputs rebuilt here from the seeds of tests/campaign.py).

The sweep's validity chain is not the reference's arithmetic (squared, division-free forms, interval screens --
DESIGN.md section 7), so argmin identity is an empirical claim; this is the evidence: 5000 config-4 queries, 2000
queries whose limits cut through the candidates' range, the 500-step config-5 relaxation rollout (1500 stateful
plan() calls) and the dense config-3 grid, each held to the reference's chosen index, per-candidate categories
(CRC-32 of the category vector; the vector itself for config 3), last_check_stats and cost (1e-9 relative).
"""
import json
import os

import numpy as np
import pytest

from oracle import frenet_oracle as O
from tests import campaign, runners, scenarios

pytestmark = pytest.mark.gpu
RTOL = 1e-9      # north_star: costs / trajectory points within 1e-9 relative in fp64


def _planner(knobs, wp, **kw):
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    return BatchFrenetPlanner(CubicSpline2D(*wp), **knobs, **kw)


def _compare(tag, res, g, ids, explain=None):
    """res: SweepResult with candidates for the queries `ids` of golden store `g`."""
    n_c = g["n_cand"][ids]
    assert np.array_equal(res.n_cand, n_c), tag
    bad = []
    for j, i in enumerate(ids):
        ok = int(res.best_idx[j]) == int(g["best"][i])
        want = g["stats"][i]
        got = res.stats[j]
        ok &= np.array_equal(got[:7], want[:7]) and (want[7] < 0 or got[7] == want[7])
        ok &= campaign.crc(res.cand_cat[j, :n_c[j]]) == int(g["crc"][i])
        if ok and g["best"][i] >= 0:
            ok &= abs(res.best_cost[j] - g["cost"][i]) <= RTOL * abs(g["cost"][i])
        if not ok:
            bad.append(int(i))
    msg = ""
    if bad and explain is not None:
        msg = explain(bad[0])
    assert not bad, f"{tag}: {len(bad)} of {len(ids)} queries differ from the reference: {bad[:20]} {msg}"


def test_config4_campaign_5000_queries():
    """Campaign A: 5000 config-4 style queries.  The host-side ego -> Frenet conversion must reproduce the
    reference's Frenet state (1e-12), the sweep the reference's decisions on that state."""
    g = runners.load_golden("campaign_a.npz")
    assert len(g["best"]) == campaign.N_A
    from integrated_path_planning_b200 import CubicSpline2D
    from integrated_path_planning_b200.frenet_host import CoordinateConverter, ego_to_frenet
    from integrated_path_planning_b200.types import EgoVehicleState
    spline = CubicSpline2D(*scenarios.STRAIGHT_60)
    pl = _planner(scenarios.S1_KNOBS, scenarios.STRAIGHT_60)
    chunk = 1000
    found = 0
    for lo in range(0, campaign.N_A, chunk):
        ids = np.arange(lo, min(lo + chunk, campaign.N_A))
        dyn = np.empty((len(ids), 50, 51, 2))
        fs = np.empty((len(ids), 6))
        for j, i in enumerate(ids):
            ego, dyn[j] = campaign.query_a(int(i))
            fs[j] = ego_to_frenet(CoordinateConverter(spline), EgoVehicleState(*ego), 0.0)
        np.testing.assert_allclose(fs, g["fs"][ids], rtol=1e-12, atol=1e-15, err_msg="ego -> Frenet")
        res = pl.plan_batch(g["fs"][ids], campaign.TARGET_SPEED, dynamic_obstacles=dyn, want_candidates=True)
        _compare("campaign A", res, g, ids)
        found += int((res.best_idx >= 0).sum())
    assert found == int((g["best"] >= 0).sum()) and found > 1000


def test_limits_campaign_2000_queries():
    """Campaign B: limits (speed, acceleration, curvature, lateral acceleration, road width) drawn through the range
    the candidates take, on three paths, including stop-target queries with the stop-distance directive."""
    g = runners.load_golden("campaign_b.npz")
    assert len(g["best"]) == campaign.N_B
    qs = [campaign.query_b(i) for i in range(campaign.N_B)]
    cats_seen = np.zeros(8, dtype=np.int64)
    for path in campaign.PATH_NAMES:
        for road in (2.7, 1.1):
            ids = np.array([i for i, q in enumerate(qs) if q["path"] == path and q["road"] == road])
            pl = _planner(campaign.knobs_b(road), campaign.PATHS[path])
            limits = np.stack([pl.resolve_limits(qs[i]["overrides"]) for i in ids])
            msd = np.array([np.nan if qs[i]["msd"] is None else qs[i]["msd"] for i in ids])
            res = pl.plan_batch(np.stack([qs[i]["fs"] for i in ids]), np.array([qs[i]["target"] for i in ids]),
                                dynamic_obstacles=np.stack([qs[i]["dyn"] for i in ids]), limits=limits,
                                max_stop_distance=msd, want_candidates=True)

            def explain(i, pl=pl, path=path, road=road):
                q = qs[i]
                orc = O.OraclePlanner(O.Spline2D(*campaign.PATHS[path]), O.Knobs(**campaign.knobs_b(road)))
                ref = orc.plan_frenet(tuple(q["fs"]), np.empty((0, 2)), q["dyn"], q["target"], q["overrides"], None, q["msd"])
                j = int(np.nonzero(ids == i)[0][0])
                got = res.cand_cat[j, :len(ref.categories)].astype(np.int8)
                d = np.nonzero(got != ref.categories)[0]
                return f"query {i} ({path}, road {road}): vs oracle port: candidates {d[:8]} got {got[d[:8]]} want {ref.categories[d[:8]]}"

            _compare(f"campaign B {path}/{road}", res, g, ids, explain)
            cats_seen += res.stats.sum(axis=0)
    assert np.all(cats_seen[:6] > 0), cats_seen            # every validity category is exercised


def test_config5_rollout_500_steps():
    """Campaign C = BASELINE config 5: 500 steps x (NORMAL, CAUTION, EMERGENCY) through the stateful plan() API
    (ego -> Frenet with the nearest-point cache, `_last_kappa` fed back), against the reference's 1500 answers."""
    from integrated_path_planning_b200 import CubicSpline2D, FrenetPlanner
    g = runners.load_golden("campaign_c.npz")
    assert len(g["best"]) == 3 * campaign.N_C_STEPS
    cu = FrenetPlanner(CubicSpline2D(*campaign.C_PATH), **scenarios.S1_KNOBS)
    seen_fs = []
    inner = cu.plan_from_frenet

    def capture(frenet_state, *a, **k):
        seen_fs.append(np.array(frenet_state, dtype=float))
        return inner(frenet_state, *a, **k)

    cu.plan_from_frenet = capture
    n, bad, counts = 0, [], set()
    for step, ego, dyn, static in campaign.rollout_c():
        for target, ovr, msd in campaign.plans_c():
            st = np.empty((0, 2)) if static is None else static
            assert cu._last_kappa == pytest.approx(float(g["kappa_in"][n]), rel=RTOL, abs=1e-15), n
            cu.plan(runners._Ego(*ego), st, dyn, target, ovr, None, msd, _want_candidates=True)
            res = cu.last_result
            np.testing.assert_allclose(seen_fs[-1], g["fs"][n], rtol=RTOL, atol=1e-12, err_msg=f"call {n}: ego -> Frenet")
            n_c = int(g["n_cand"][n])
            want = g["stats"][n]
            ok = int(res.n_cand[0]) == n_c and int(res.best_idx[0]) == int(g["best"][n])
            ok = ok and np.array_equal(res.stats[0][:7], want[:7]) and (want[7] < 0 or res.stats[0][7] == want[7])
            ok = ok and campaign.crc(res.cand_cat[0, :n_c]) == int(g["crc"][n])
            if ok and g["best"][n] >= 0:
                ok = abs(res.best_cost[0] - g["cost"][n]) <= RTOL * abs(g["cost"][n])
            if not ok:
                bad.append(n)
            counts.add(n_c)
            n += 1
    assert not bad, f"config 5: {len(bad)} of {n} plan() calls differ from the reference: {bad[:20]}"
    assert {1261, 843, 216} <= counts


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("kernel", ["pairs", "items"])
def test_config3_dense_grid_against_the_reference(variant, kernel):
    """Campaign D = BASELINE config 3 at its stated size, BOTH sweep kernels against one recorded reference run
    (59.8 s of NumPy): per-candidate categories, costs, winner."""
    name = f"config3_v{variant}.npz"
    if not os.path.exists(os.path.join(runners.GOLDEN_DIR, name)):
        pytest.skip(f"{name} not recorded")
    g = runners.load_golden(name)
    c = campaign.config3(variant)
    pl = _planner(c["knobs"], c["waypoints"])
    pl.engine                                  # the handle exists before the option is switched
    with runners.fot_env(FOT_SWEEP=kernel):
        res = pl.plan_batch(c["fs"][None], c["target"], distribution=c["dist"][None], want_candidates=True)
    n_c = len(g["cats"])
    assert int(res.n_cand[0]) == n_c == 66563
    mism = np.nonzero(res.cand_cat[0, :n_c] != g["cats"])[0]
    assert mism.size == 0, (mism[:10], res.cand_cat[0, mism[:10]], g["cats"][mism[:10]])
    np.testing.assert_allclose(res.cand_cost[0, :n_c], g["costs"], rtol=RTOL, atol=0)
    assert int(res.best_idx[0]) == int(g["best"])
    want = g["stats"]
    assert np.array_equal(res.stats[0][:7], want[:7])
    if int(g["best"]) >= 0:
        assert abs(res.best_cost[0] - float(g["cost"])) <= RTOL * abs(float(g["cost"]))
        series = res.series(0)
        for s in runners.SERIES:
            np.testing.assert_allclose(series[s], g["w_" + s], rtol=RTOL, atol=runners.ATOL, err_msg=s)


def test_threshold_margin_histogram():
    """SURVEY.md section 7: log how close the checked quantities come to their limits.  For a sample of campaign A and
    B queries the oracle port (which reproduces the reference bit for bit) reports, per candidate and test, the
    smallest relative distance to the limit; the histogram goes to gpurun_out/threshold_margins.json.  The CUDA
    chain differs from the reference's values by ~1e-15 relative; the campaign's categories are identical, and this
    shows how much room there was."""
    edges = 10.0 ** np.arange(-16, 1)
    hist = {}
    smallest = {}

    def add(m):
        for name, v in m.items():
            v = v[np.isfinite(v)]
            h = np.histogram(np.clip(v, 1e-16, 0.999), bins=edges)[0]
            hist[name] = hist.get(name, 0) + h
            if len(v):
                smallest[name] = min(smallest.get(name, np.inf), float(v.min()))

    orc = O.OraclePlanner(O.Spline2D(*scenarios.STRAIGHT_60), O.Knobs(**scenarios.S1_KNOBS))
    for i in range(0, 40):
        ego, dyn = campaign.query_a(i)
        orc.reset_ego_curvature()
        orc.plan(ego, np.empty((0, 2)), dyn, campaign.TARGET_SPEED)
        add(O.threshold_margins(orc.k, orc.last_candidates))
    for i in range(0, 120):
        q = campaign.query_b(i)
        ob = O.OraclePlanner(O.Spline2D(*campaign.PATHS[q["path"]]), O.Knobs(**campaign.knobs_b(q["road"])))
        ob.plan_frenet(tuple(q["fs"]), np.empty((0, 2)), q["dyn"], q["target"], q["overrides"], None, q["msd"])
        add(O.threshold_margins(ob.k, ob.last_candidates, q["overrides"]))
    report = {"bins_log10_lower_edge": list(range(-16, 0)),
              "histogram": {k: v.tolist() for k, v in hist.items()}, "smallest_margin": smallest,
              "sample": "campaign A queries 0-39 and campaign B queries 0-119 (oracle port)"}
    os.makedirs("gpurun_out", exist_ok=True)
    with open(os.path.join("gpurun_out", "threshold_margins.json"), "w") as f:
        json.dump(report, f, indent=1)
    print("\nthreshold margins (smallest relative distance to a limit):", {k: f"{v:.2e}" for k, v in smallest.items()})
    assert sum(int(np.sum(h)) for h in hist.values()) > 50000
