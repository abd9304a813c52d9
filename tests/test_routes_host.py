"""Host side of multi-route batches (no GPU): the fot_route_t layout, the new symbols, the checks of `route` that run
before anything reaches the device, and the route grouping of RoutedCoordinateConverter's host path."""
import ctypes
import os
import re

import numpy as np
import pytest

from tests import scenarios

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_route_struct_and_symbols():
    from integrated_path_planning_b200 import _lib
    assert ctypes.sizeof(_lib.FotRoute) == 8 + 9 * 8               # int32 nx (padded) + ten pointers
    header = open(os.path.join(ROOT, "include", "fot.h")).read()
    for name in ("fot_add_route", "fot_set_routes"):
        assert re.search(r"^\s*int\s+%s\s*\(" % name, header, flags=re.M), name
        assert name in {n for n, _, _ in _lib.SYMBOLS}
        assert hasattr(_lib.load(), name)
    assert "fot_route_t" in header


def test_route_array_checks():
    from integrated_path_planning_b200.engine import route_array
    assert route_array(None, 4, 3) is None
    np.testing.assert_array_equal(route_array(2, 4, 3), [2, 2, 2, 2])
    a = route_array(np.array([0, 1, 2, 1], dtype=np.int64), 4, 3)
    assert a.dtype == np.int32 and a.flags.c_contiguous
    for bad in (3, -1, [0, 1, 2], [[0, 1], [2, 0]], [0.0, 1.0, 2.0, 1.0], 1.0, True, np.array([0, 1, 3, 0]), "0"):
        with pytest.raises(ValueError):
            route_array(bad, 4, 3)


def _planner():
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    pl = BatchFrenetPlanner(CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    assert pl.add_route(CubicSpline2D(*scenarios.arc_waypoints())) == 1
    return pl


def test_bad_route_raises_before_the_device():
    """The planner on a machine without a GPU: a bad `route` is a ValueError, not a device error, so it is checked
    first (the engine, which needs the device, is never created)."""
    from integrated_path_planning_b200 import DeviceBatch, _lib
    pl = _planner()
    fs = np.zeros((3, 6))
    fs[:, 1] = 2.0
    for bad in (2, [0, 1], [0, 1, 5], [0.5, 1, 0], [-1, 0, 0]):
        with pytest.raises(ValueError):
            pl.plan_batch(fs, 6.0, route=bad)
        with pytest.raises(ValueError):
            pl.plan_batch_from_ego(np.zeros((3, 5)), 6.0, route=bad)
        with pytest.raises(ValueError):
            DeviceBatch(pl, fs, 6.0, None, _lib.FOT_DYN_NONE, route=bad)
    assert pl._engine is None


def test_add_route_refuses_a_path_without_coefficients():
    pl = _planner()
    with pytest.raises(TypeError):
        pl.add_route(object())
    assert len(pl.routes) == 2 and pl._engine is None


def test_routed_converter_groups_rows_by_route_on_the_host():
    """Without an engine every row is searched on the host by its own route's converter: results, caches and the row
    counts equal one BatchCoordinateConverter per route."""
    from integrated_path_planning_b200 import CubicSpline2D
    from integrated_path_planning_b200.frenet_host import BatchCoordinateConverter, RoutedCoordinateConverter
    rng = np.random.default_rng(3)
    paths = [CubicSpline2D(*scenarios.STRAIGHT_60), CubicSpline2D(*scenarios.arc_waypoints()),
             CubicSpline2D(*scenarios.s_curve_waypoints())]
    n = 30
    route = rng.integers(0, 3, n)
    conv = RoutedCoordinateConverter(paths, route)
    per = {r: BatchCoordinateConverter(p, int((route == r).sum())) for r, p in enumerate(paths)}
    for step in range(3):
        x, y = rng.uniform(0, 50, n), rng.uniform(-3, 12, n)
        got = conv.reference_points(np.arange(n), x, y)
        for r, c in per.items():
            rows = np.nonzero(route == r)[0]
            want = c.reference_points(np.arange(len(rows)), x[rows], y[rows])
            for a, b in zip(got, want):
                np.testing.assert_array_equal(a[rows], b)
            np.testing.assert_array_equal(conv.prev_s[rows], c.prev_s)
    assert conv.device_rows == 0 and conv.host_rows == 0


def test_routed_converter_checks_its_routes():
    """A negative or too large id, a non-integer or a 2-D route is a ValueError, never a wrap-around into the list."""
    from integrated_path_planning_b200 import CubicSpline2D
    from integrated_path_planning_b200.frenet_host import RoutedCoordinateConverter
    paths = [CubicSpline2D(*scenarios.STRAIGHT_60), CubicSpline2D(*scenarios.arc_waypoints())]
    for bad in ([0, -1], [0, 2], [0.0, 1.0], [[0, 1]]):
        with pytest.raises(ValueError):
            RoutedCoordinateConverter(paths, bad)
    assert list(RoutedCoordinateConverter(paths, [1, 0]).route) == [1, 0]
