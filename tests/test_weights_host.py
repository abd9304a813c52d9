"""CPU: the host side of the cost-weight sweeps (fot_weighted_t, weight parsing, SweepResult.under_weights)."""
import ctypes
import os
import re

import numpy as np
import pytest

from tests import scenarios

import integrated_path_planning_b200 as ipp
from integrated_path_planning_b200 import _lib
from integrated_path_planning_b200.batch import _weight_table
from integrated_path_planning_b200.engine import SweepResult
from integrated_path_planning_b200.types import SERIES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_weighted_struct_layout_and_constants_match_header():
    assert ctypes.sizeof(_lib.FotWeighted) == 2 * 4 + 5 * 8          # int32 n_w, per_query + five pointers
    assert [name for name, _ in _lib.FotWeighted._fields_] == ["n_w", "per_query", "weights", "idx", "cost", "len", "series"]
    header = open(os.path.join(ROOT, "include", "fot.h")).read()
    assert int(re.search(r"#define FOT_MAX_WEIGHT_SETS (\d+)", header).group(1)) == _lib.FOT_MAX_WEIGHT_SETS == 256
    # an addition that changes no existing struct or entry point: same version, next minor revision
    assert int(re.search(r"#define FOT_ABI_VERSION (\d+)", header).group(1)) == _lib.FOT_ABI_VERSION == 8
    assert int(re.search(r"#define FOT_ABI_MINOR (\d+)", header).group(1)) == _lib.FOT_ABI_MINOR == 1
    assert _lib.COST_WEIGHT_KEYS == ("k_j", "k_t", "k_d", "k_s_dot", "k_lat", "k_lon")
    fields = re.search(r"typedef struct fot_weighted \{(.*?)\} fot_weighted_t;", header, re.S).group(1)
    assert re.findall(r"^\s*(?:const\s+)?\w+\*?\s+\*?(\w+);", fields, re.M) == ["n_w", "per_query", "weights", "idx", "cost", "len", "series"]
    # the ranked struct is unchanged by this version
    assert ctypes.sizeof(_lib.FotRanked) == 8 + 4 * 8
    assert int(re.search(r"#define FOT_MAX_RANKED (\d+)", header).group(1)) == _lib.FOT_MAX_RANKED == 32
    for name in ("fot_select_weighted", "fot_cost_terms", "fot_abi_minor"):
        assert name in [s[0] for s in _lib.SYMBOLS] and re.search(rf"int {name}\(", header)


def _planner():
    return ipp.FrenetPlanner(ipp.CubicSpline2D(*scenarios.STRAIGHT_60), **dict(scenarios.S1_KNOBS, k_d=2.5, k_lon=0.5))


def test_weight_dicts_take_the_planners_own_values_for_missing_keys():
    pl = _planner()
    w = pl.cost_weight_table([{"k_j": 0.1}, {}, {"k_lat": 3.0, "k_s_dot": 0.0}])
    own = [pl.k_j, pl.k_t, pl.k_d, pl.k_s_dot, pl.k_lat, pl.k_lon]
    assert w.dtype == np.float64 and w.shape == (3, 6)
    assert w[0].tolist() == [0.1] + own[1:]
    assert w[1].tolist() == own == [1.0, 1.0, 2.5, 1.0, 1.0, 0.5]
    assert w[2].tolist() == [1.0, 1.0, 2.5, 0.0, 3.0, 0.5]
    assert pl.cost_weight_table({"k_d": 1.0}).tolist() == [[1.0, 1.0, 1.0, 1.0, 1.0, 0.5]]
    arr = np.arange(12.0).reshape(2, 6)
    assert np.array_equal(pl.cost_weight_table(arr), arr)
    assert np.array_equal(pl.cost_weight_table(arr.tolist()), arr)


def test_bad_weights_are_rejected_before_planning():
    pl = _planner()
    ego = ipp.EgoVehicleState(5.0, 0.0, 0.0, 5.0, 0.0)
    for bad in ([{"k_jerk": 1.0}], np.ones((0, 6)), np.ones((_lib.FOT_MAX_WEIGHT_SETS + 1, 6)), np.ones((2, 5)),
                np.ones(6), None, []):
        with pytest.raises(ValueError):
            pl.plan_under_weights(ego, np.empty((0, 2)), weights=bad)
    assert pl._engine is None and pl.last_check_stats is None


def test_weight_table_shapes():
    w, pq = _weight_table(np.ones((3, 6)), n_q=5)
    assert pq == 0 and w.shape == (3, 6) and w.flags.c_contiguous
    w, pq = _weight_table(np.ones((5, 1, 6)), n_q=5)
    assert pq == 1 and w.shape == (5, 1, 6)
    assert _weight_table(None, n_q=5) == (None, 0)
    for bad in (np.ones((4, 1, 6)), np.ones((3, 7)), np.ones(6), np.ones((0, 6)), np.ones((5, 257, 6)), np.ones((2, 3, 4, 6))):
        with pytest.raises(ValueError):
            _weight_table(bad, n_q=5)


def _result(with_series=True):
    n_q, n_w, n_t = 2, 3, 7
    rng = np.random.default_rng(0)
    res = SweepResult(best_idx=np.array([5, -1], np.int32), best_cost=np.array([1.5, np.inf]),
                      stats=np.zeros((n_q, 8), np.int32), winner_len=np.array([6, 0], np.int32),
                      winner=rng.normal(size=(n_q, 15, n_t)))
    res.w_idx = np.array([[5, -1, 9], [-1, -1, -1]], np.int32)
    res.w_cost = np.array([[1.5, np.inf, 0.25], [np.inf] * 3])
    if with_series:
        res.w_len = np.array([[6, 0, 3], [0, 0, 0]], np.int32)
        res.w_series = rng.normal(size=(n_q, n_w, 15, n_t))
    return res


def test_under_weights_one_entry_per_weighting():
    res = _result()
    ws = res.under_weights(0)
    assert len(ws) == 3 and ws[1] is None
    assert [w["index"] for w in (ws[0], ws[2])] == [5, 9]
    assert [w["cost"] for w in (ws[0], ws[2])] == [1.5, 0.25] and isinstance(ws[2]["cost"], np.float64)
    for w, e in ((0, ws[0]), (2, ws[2])):
        n = int(res.w_len[0, w])
        assert set(e["series"]) == set(SERIES) and len(e["series"]["x"]) == n
        for j, name in enumerate(SERIES):
            assert np.array_equal(e["series"][name], res.w_series[0, w, j, :n])
    ws[0]["series"]["t"][0] = 123.0                                # a copy, not a view into the result
    assert res.w_series[0, 0, 0, 0] != 123.0
    assert res.under_weights(1) == [None, None, None]


def test_under_weights_without_series():
    res = _result(with_series=False)
    ws = res.under_weights(0)
    assert ws[1] is None and ws[0]["series"] is None and ws[2]["index"] == 9
