"""CPU: the host side of the ranked alternatives (fot_ranked_t, SweepResult.alternatives)."""
import ctypes
import os
import re

import numpy as np
import pytest

from tests import scenarios

import integrated_path_planning_b200 as ipp
from integrated_path_planning_b200 import _lib
from integrated_path_planning_b200.engine import SweepResult
from integrated_path_planning_b200.types import SERIES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ranked_struct_layout_and_limit_match_header():
    assert ctypes.sizeof(_lib.FotRanked) == 8 + 4 * 8           # int32 k (padded to 8) + four pointers
    assert [name for name, _ in _lib.FotRanked._fields_] == ["k", "idx", "cost", "len", "series"]
    header = open(os.path.join(ROOT, "include", "fot.h")).read()
    assert int(re.search(r"#define FOT_MAX_RANKED (\d+)", header).group(1)) == _lib.FOT_MAX_RANKED == 32
    assert int(re.search(r"#define FOT_ABI_VERSION (\d+)", header).group(1)) == _lib.FOT_ABI_VERSION == 8


def _result(k=4, n_t=7, with_series=True):
    n_q = 3
    rng = np.random.default_rng(0)
    res = SweepResult(best_idx=np.array([5, -1, 2], np.int32), best_cost=np.array([1.5, np.inf, 0.25]),
                      stats=np.zeros((n_q, 8), np.int32), winner_len=np.array([6, 0, 7], np.int32),
                      winner=rng.normal(size=(n_q, 15, n_t)))
    res.rank_idx = np.array([[5, 9, 1, -1], [-1, -1, -1, -1], [2, 3, 4, 0]], np.int32)[:, :k]
    res.rank_cost = np.array([[1.5, 1.5, 2.0, np.inf], [np.inf] * 4, [0.25, 0.5, 0.75, 1.0]])[:, :k]
    if with_series:
        res.rank_len = np.array([[6, 3, 7, 0], [0] * 4, [7, 7, 2, 5]], np.int32)[:, :k]
        res.rank_series = rng.normal(size=(n_q, k, 15, n_t))
    return res


def test_alternatives_in_rank_order_truncated_to_kept_length():
    res = _result()
    alts = res.alternatives(0)
    assert [a["index"] for a in alts] == [5, 9, 1]                  # stops at the first padded rank
    assert [a["cost"] for a in alts] == [1.5, 1.5, 2.0]
    assert all(isinstance(a["cost"], np.float64) for a in alts)
    for r, a in enumerate(alts):
        n = int(res.rank_len[0, r])
        assert set(a["series"]) == set(SERIES)
        for j, name in enumerate(SERIES):
            assert np.array_equal(a["series"][name], res.rank_series[0, r, j, :n])
        assert len(a["series"]["x"]) == n
    a0 = alts[0]["series"]["t"]
    a0[0] = 123.0                                                   # a copy, not a view into the result
    assert res.rank_series[0, 0, 0, 0] != 123.0
    assert res.alternatives(1) == []
    assert [a["index"] for a in res.alternatives(2)] == [2, 3, 4, 0]  # k entries when all are feasible


def test_alternatives_without_series():
    res = _result(with_series=False)
    alts = res.alternatives(2)
    assert [a["index"] for a in alts] == [2, 3, 4, 0]
    assert all(a["series"] is None for a in alts)


def test_plan_alternatives_rejects_k_outside_range_before_planning():
    pl = ipp.FrenetPlanner(ipp.CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    ego = ipp.EgoVehicleState(5.0, 0.0, 0.0, 5.0, 0.0)
    for k in (0, -1, _lib.FOT_MAX_RANKED + 1):
        with pytest.raises(ValueError):
            pl.plan_alternatives(ego, np.empty((0, 2)), k=k)
    assert pl._engine is None and pl.last_check_stats is None
