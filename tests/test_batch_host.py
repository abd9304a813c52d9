"""CPU: how a batch reaches the C ABI -- the input normaliser (query_arrays), the fot_batch_t / fot_result_t fillers,
the winner block's field list and SweepResult.blank -- and malformed input refused before any device work."""
import dataclasses

import numpy as np
import pytest
import torch

from tests import scenarios

import integrated_path_planning_b200 as ipp
from integrated_path_planning_b200 import _lib
from integrated_path_planning_b200.batch import DeviceBatch, WinnerBlock
from integrated_path_planning_b200.engine import (SweepResult, fot_batch, fot_result, query_arrays, speed_grid_batch,
                                                  winner_fields)

D_T_S = scenarios.S1_KNOBS["d_t_s"]
N_Q = 3
LIMITS = [10.0, 2.0, 0.2, 3.0]
host_ptr = lambda a: a.ctypes.data


@pytest.fixture
def frenet():
    return np.arange(6.0 * N_Q).reshape(N_Q, 6) / 10.0


@pytest.fixture
def planner():
    return ipp.BatchFrenetPlanner(ipp.CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)


def _arrays(frenet, **kw):
    args = dict(target_speed=6.0, limits=LIMITS, stop_dist=None, static=None, dyn=None, dyn_mode=_lib.FOT_DYN_NONE)
    args.update(kw)
    return query_arrays(frenet, args["target_speed"], args["limits"], args["stop_dist"], args["static"], args["dyn"],
                        args["dyn_mode"], D_T_S)


def _is_f64c(a):
    return a.dtype == np.float64 and a.flags.c_contiguous


def test_query_arrays_broadcasts_and_defaults(frenet):
    q = _arrays(frenet.tolist(), dyn=np.ones((N_Q, 1, 2, 4, 2)))          # a dyn with FOT_DYN_NONE is ignored
    assert all(_is_f64c(a) for a in (q.frenet, q.target, q.limits, q.stop))
    assert np.array_equal(q.frenet, frenet)
    assert q.target.tolist() == [6.0] * N_Q and q.limits.tolist() == [LIMITS] * N_Q and np.isnan(q.stop).all()
    want_grid, want_n_v = speed_grid_batch(np.full(N_Q, 6.0), D_T_S)
    assert np.array_equal(q.v_grid, want_grid) and np.array_equal(q.n_v, want_n_v) and q.n_v.dtype == np.int32
    assert q.static is None and not q.static_per_query and q.dyn is None and q.dyn_mode == _lib.FOT_DYN_NONE

    target = np.array([6.0, 3.0, 0.0])
    q = _arrays(frenet, target_speed=target, stop_dist=5.0, limits=np.tile(LIMITS, (N_Q, 1)))
    assert np.array_equal(q.target, target) and q.stop.tolist() == [5.0] * N_Q and q.limits.shape == (N_Q, 4)
    want_grid, want_n_v = speed_grid_batch(target, D_T_S)
    assert np.array_equal(q.v_grid, want_grid) and np.array_equal(q.n_v, want_n_v)

    wall = scenarios.wall(x=30.0)
    q = _arrays(frenet, static=wall.tolist())
    assert _is_f64c(q.static) and np.array_equal(q.static, wall) and not q.static_per_query
    q = _arrays(frenet, static=np.stack([wall] * N_Q))
    assert q.static.shape == (N_Q,) + wall.shape and q.static_per_query
    assert _arrays(frenet, static=np.empty((0, 2))).static is None

    q = _arrays(frenet, dyn=np.ones((N_Q, 1, 2, 4, 2), dtype=np.float32), dyn_mode=_lib.FOT_DYN_SINGLE)
    assert _is_f64c(q.dyn) and q.dyn.shape == (N_Q, 1, 2, 4, 2) and q.dyn_mode == _lib.FOT_DYN_SINGLE
    t = torch.ones((N_Q, 2, 2, 4, 2), dtype=torch.float64)
    q = _arrays(frenet, dyn=t, dyn_mode=_lib.FOT_DYN_DISTRIBUTION)
    assert q.dyn is t                                                      # a tensor is left where it is


@pytest.mark.parametrize("dyn", [np.ones((N_Q, 2, 4, 2)), np.ones((N_Q + 1, 1, 2, 4, 2)), np.ones((N_Q, 1, 2, 4, 3)),
                                 torch.ones((N_Q, 1, 2, 4, 2), dtype=torch.float32)],
                         ids=["ndim", "first_dim", "last_dim", "dtype"])
def test_query_arrays_rejects_malformed_dyn(frenet, dyn):
    with pytest.raises(ValueError, match="dyn"):
        _arrays(frenet, dyn=dyn, dyn_mode=_lib.FOT_DYN_SINGLE)


@pytest.mark.parametrize("static", [np.ones((N_Q - 1, 5, 2)), np.ones((5, 3)), np.ones(4), np.ones((N_Q, 5, 3))],
                         ids=["per_query_first_dim", "last_dim", "ndim", "per_query_last_dim"])
def test_query_arrays_rejects_malformed_static(frenet, static):
    with pytest.raises(ValueError, match="static"):
        _arrays(frenet, static=static)


def test_fot_batch_fills_every_field(frenet):
    dyn = np.ones((N_Q, 2, 3, 4, 2))
    q = _arrays(frenet, static=np.ones((N_Q, 5, 2)), dyn=dyn, dyn_mode=_lib.FOT_DYN_DISTRIBUTION)
    b = fot_batch(q, host_ptr)
    assert (b.n_q, b.n_v_max) == (N_Q, q.v_grid.shape[1])
    for field, a in (("frenet", q.frenet), ("target_speed", q.target), ("limits", q.limits), ("stop_dist", q.stop),
                     ("v_grid", q.v_grid), ("n_v", q.n_v), ("static_obs", q.static), ("dyn", q.dyn)):
        assert getattr(b, field) == a.ctypes.data, field
    assert (b.n_static, b.static_per_query) == (5, 1)
    assert (b.S, b.P, b.T_obs, b.dyn_mode) == (2, 3, 4, _lib.FOT_DYN_DISTRIBUTION)

    b = fot_batch(_arrays(frenet, static=np.ones((5, 2))), host_ptr)
    assert b.static_obs is not None and (b.n_static, b.static_per_query) == (5, 0)
    assert b.dyn is None and (b.S, b.P, b.T_obs, b.dyn_mode) == (0, 0, 0, _lib.FOT_DYN_NONE)
    b = fot_batch(_arrays(frenet), host_ptr)
    assert b.static_obs is None and b.n_static == 0

    # the device path: the same fields from copies of the arrays (here CPU tensors), through their data_ptr()
    copies = {k: torch.from_numpy(getattr(q, k).copy()) for k in ("frenet", "target", "limits", "stop", "v_grid",
                                                                   "n_v", "static", "dyn")}
    b = fot_batch(dataclasses.replace(q, **copies), torch.Tensor.data_ptr)
    assert b.frenet == copies["frenet"].data_ptr() and b.dyn == copies["dyn"].data_ptr()
    assert b.static_obs == copies["static"].data_ptr() and (b.S, b.P, b.T_obs, b.n_static) == (2, 3, 4, 5)


def _winner_arrays(n_q=N_Q, n_t=7):
    return {name: torch.zeros((n_q, *shape), dtype=dt).numpy() for name, dt, shape in winner_fields(n_t)}


def test_fot_result_fills_the_winner_block_and_candidate_table():
    arrays = _winner_arrays()
    r = fot_result(arrays, host_ptr)
    for name in ("best_idx", "best_cost", "stats", "winner_len", "winner"):
        assert getattr(r, name) == arrays[name].ctypes.data, name
    assert r.cand_cat is None and r.cand_cost is None and r.cand_stride == 0 and r.winner_samples == 0

    arrays.update(cand_cat=np.zeros((N_Q, 11), np.uint8), cand_cost=np.zeros((N_Q, 11)))
    r = fot_result(arrays, host_ptr, winner_samples=2)
    assert r.cand_cat == arrays["cand_cat"].ctypes.data and r.cand_cost == arrays["cand_cost"].ctypes.data
    assert r.cand_stride == 11 and r.winner_samples == 2
    arrays["cand_cost"] = None                                            # categories alone (cost weightings)
    r = fot_result(arrays, host_ptr)
    assert r.cand_cat == arrays["cand_cat"].ctypes.data and r.cand_cost is None and r.cand_stride == 11

    # raw addresses, as the peer-memory mirror passes them
    r = fot_result({name: 4096 * (i + 1) for i, (name, _, _) in enumerate(winner_fields(0))}, int)
    assert [r.best_idx, r.winner_len, r.stats, r.best_cost, r.winner] == [4096, 8192, 12288, 16384, 20480]


def test_winner_fields_are_the_winner_block_layout():
    assert [name for name, _, _ in winner_fields(7)] == ["best_idx", "winner_len", "stats", "best_cost", "winner"]
    blk = WinnerBlock(4, 7)
    assert blk.sections == winner_fields(7)
    assert list(blk.offsets) == [name for name, _, _ in winner_fields(7)]
    for name, dt, shape in winner_fields(7):
        assert blk.views[name].dtype == dt and tuple(blk.views[name].shape) == (4, *shape)


def _full_result(n_q=4, k=3, n_w=2, n_t=7, stride=11):
    rng = np.random.default_rng(0)
    res = SweepResult(best_idx=np.arange(n_q, dtype=np.int32), best_cost=rng.normal(size=n_q),
                      stats=np.ones((n_q, 8), np.int32), winner_len=np.full(n_q, 5, np.int32),
                      winner=rng.normal(size=(n_q, 15, n_t)), cand_cat=np.ones((n_q, stride), np.uint8),
                      cand_cost=rng.normal(size=(n_q, stride)), n_cand=np.full(n_q, stride))
    res.rank_idx, res.rank_cost = np.ones((n_q, k), np.int32), rng.normal(size=(n_q, k))
    res.rank_len, res.rank_series = np.full((n_q, k), 4, np.int32), rng.normal(size=(n_q, k, 15, n_t))
    res.w_idx, res.w_cost = np.ones((n_q, n_w), np.int32), rng.normal(size=(n_q, n_w))
    res.w_len, res.w_series = np.full((n_q, n_w), 4, np.int32), rng.normal(size=(n_q, n_w, 15, n_t))
    res.cost_terms = rng.normal(size=(n_q, stride, 5))
    return res


def test_blank_sets_exactly_the_failed_rows_outputs():
    res, ref = _full_result(), _full_result()
    rows = np.array([False, True, False, True])
    res.blank(rows)
    blanked = {"best_idx": -1, "best_cost": np.inf, "stats": 0, "winner_len": 0, "rank_idx": -1, "rank_cost": np.inf,
               "rank_len": 0, "w_idx": -1, "w_cost": np.inf, "w_len": 0}
    for f in dataclasses.fields(SweepResult):
        got, want = getattr(res, f.name), getattr(ref, f.name)
        if f.name in blanked:
            assert (got[rows] == blanked[f.name]).all() and np.array_equal(got[~rows], want[~rows]), f.name
        elif f.name == "cost_terms":
            assert np.isnan(got[rows]).all() and np.array_equal(got[~rows], want[~rows])
        else:                                                             # series, candidate table, counts: untouched
            assert np.array_equal(got, want, equal_nan=True), f.name

    plain = SweepResult(best_idx=np.zeros(2, np.int32), best_cost=np.zeros(2), stats=np.ones((2, 8), np.int32),
                        winner_len=np.ones(2, np.int32), winner=np.ones((2, 15, 3)))
    plain.blank([1])                                                      # without the optional outputs
    assert plain.best_idx.tolist() == [0, -1] and plain.best_cost.tolist() == [0.0, np.inf]
    assert plain.stats[1].sum() == 0 and plain.winner_len.tolist() == [1, 0] and (plain.winner == 1.0).all()
    assert plain.rank_idx is None and plain.w_idx is None and plain.cost_terms is None


def test_malformed_batches_are_rejected_before_the_device_is_used(planner, frenet):
    per_query = np.stack([scenarios.wall(x=30.0)] * (N_Q - 1))             # one query short
    with pytest.raises(ValueError, match="static"):
        planner.plan_batch(frenet, 6.0, static_obstacles=per_query)
    with pytest.raises(ValueError, match="static"):
        planner.plan_batch(frenet, 6.0, static_obstacles=np.ones((5, 3)), top_k=4)
    with pytest.raises(ValueError, match="static"):
        planner.plan_batch_from_ego(np.zeros((N_Q, 5)), 6.0, static_obstacles=per_query)
    with pytest.raises(ValueError, match="dyn"):
        planner.plan_batch(frenet, 6.0, distribution=np.ones((N_Q, 2, 3, 4)))
    for bad in (np.ones((N_Q, 1, 2, 4)), np.ones((N_Q + 1, 1, 2, 4, 2)), torch.ones((N_Q, 1, 2, 4, 2))):
        with pytest.raises(ValueError, match="dyn"):
            DeviceBatch(planner, frenet, 6.0, bad, _lib.FOT_DYN_SINGLE)
    with pytest.raises(ValueError, match="static"):
        DeviceBatch(planner, frenet, 6.0, None, _lib.FOT_DYN_NONE, static_obstacles=per_query)
    assert planner._engine is None
