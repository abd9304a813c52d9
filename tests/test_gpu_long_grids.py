"""GPU: time grids longer than NumPy's 128-element pairwise block run the sample-major fot_sweep_items, up to its limit
of one thread per sample in a 320-thread block; shapes beyond what it takes are refused with FOT_ERR_TOO_LARGE."""
import numpy as np
import pytest

from oracle import frenet_oracle as O
from tests import runners, scenarios

pytestmark = pytest.mark.gpu

LONG_STRAIGHT = (np.linspace(0.0, 240.0, 13).tolist(), [0.0] * 13)


def _knobs(min_t, max_t):
    return dict(scenarios.S1_KNOBS, dt=0.05, min_t=min_t, max_t=max_t, d_road_w=0.9, d_t_s=3.0)


def _planner(knobs):
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    return BatchFrenetPlanner(CubicSpline2D(*LONG_STRAIGHT), **knobs)


# 129 samples: one split of the pairwise sum; 199: an uneven split (96 + 103); 320: two levels (4 blocks of 80)
@pytest.mark.parametrize("min_t, max_t, n_t", [(6.0, 6.4, 129), (9.5, 9.9, 199), (15.6, 15.95, 320)])
def test_long_time_grid_matches_the_oracle(min_t, max_t, n_t):
    """Every candidate's category equals the oracle's; costs agree within 1e-9, not bit for bit, because the oracle's
    coefficient solve follows this host's BLAS order and moves by 1 ulp on some candidates (DESIGN.md section 7)."""
    knobs = _knobs(min_t, max_t)
    rng = np.random.default_rng(n_t)
    n = 6
    frenet = np.stack([rng.uniform(2, 15, n), rng.uniform(1, 7, n), rng.uniform(-1, 1, n), rng.uniform(-1, 1, n),
                       rng.normal(0, 0.2, n), rng.normal(0, 0.05, n)], axis=1)
    dyn = np.stack([scenarios.pedestrian_field(rng, 6, n_steps=n_t, dt=0.05, x_range=(10.0, 90.0), y_range=(-6.0, 6.0))
                    for _ in range(n)])
    wall = scenarios.wall(x=70.0, half=1.5, n=13)
    pl = _planner(knobs)
    assert pl.engine.n_t_max == n_t
    res = pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn, static_obstacles=wall, want_candidates=True)
    assert int(pl.engine.lib.fot_last_sweep_kind(pl.engine._h)) == 1
    orc = O.OraclePlanner(O.Spline2D(*LONG_STRAIGHT), O.Knobs(**knobs))
    n_grid = len(O.horizon_grid(orc.k)) * len(O.speed_grid(orc.k, 6.0)) * len(O.lateral_grid(orc.k))
    n_found = 0
    for i in range(n):
        ref = orc.plan_frenet(tuple(frenet[i]), wall, dyn[i], 6.0)
        n_c = len(ref.categories)
        assert n_c > n_grid, i                                     # the brake ladder is there
        assert int(res.n_cand[i]) == n_c, i
        assert np.array_equal(res.cand_cat[i, :n_c].astype(np.int8), ref.categories), i
        np.testing.assert_allclose(res.cand_cost[i, :n_c], ref.costs, rtol=runners.RTOL, atol=0, err_msg=str(i))
        assert int(res.best_idx[i]) == ref.best_index, i
        if ref.best_index < 0:
            continue
        n_found += 1
        np.testing.assert_allclose(res.best_cost[i], ref.cost, rtol=runners.RTOL, atol=0, err_msg=str(i))
        series = res.series(i)
        for s in runners.SERIES:
            assert len(series[s]) == len(ref.arrays[s]), (i, s)
            np.testing.assert_allclose(series[s], ref.arrays[s], rtol=runners.RTOL, atol=runners.ATOL, err_msg=f"{i} {s}")
    assert n_found >= n // 2
    assert res.stats[:, 6].sum() > 0                               # pedestrians or the wall hit some candidates


def test_shapes_beyond_the_sample_major_kernel_are_refused():
    """321 samples, 32769 obstacle trajectories (S*P) and 32769 static points: plan_batch raises FotError, and the
    message names the limit."""
    from integrated_path_planning_b200._lib import FotError
    frenet = np.array([[8.0, 5.0, 0.0, 0.4, 0.0, 0.0]])
    pl = _planner(_knobs(15.7, 16.0))
    assert pl.engine.n_t_max == 321
    with pytest.raises(FotError, match="time grid of 321 samples"):
        pl.plan_batch(frenet, 6.0)
    pl = _planner(_knobs(4.0, 5.0))
    dyn = scenarios.pedestrian_field(np.random.default_rng(0), 32769, n_steps=8, dt=0.05)
    with pytest.raises(FotError, match="32769 obstacle trajectories"):
        pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[None])
    with pytest.raises(FotError, match="32769 static obstacle points"):
        pl.plan_batch(frenet, 6.0, static_obstacles=scenarios.wall(x=70.0, half=1.5, n=32769))
    pl.plan_batch(frenet, 6.0, dynamic_obstacles=dyn[None, :32768])           # at the limit: no error
    assert int(pl.engine.lib.fot_last_sweep_kind(pl.engine._h)) in (1, 4)
