"""Ego state -> Frenet initial conditions, on the host (O(1) per query, stateful).

Restates reference `src/core/coordinate_converter.py:26-88` (Cartesian->Frenet formulas) and
`:202-339` (nearest point on the path with the `_prev_s` window cache), plus the spatial->time
derivative conversion of `frenet_planner.py:362-371`.  These produce the six numbers that seed
every candidate polynomial, so they follow the reference's arithmetic literally.
"""
from __future__ import annotations

import bisect
import math
from typing import Optional, Tuple

import numpy as np


def _f(v):
    """numpy 0-d / 1-element result -> scalar."""
    v = np.asarray(v)
    return v.reshape(-1)[0] if v.size == 1 else v


class CoordinateConverter:
    """Nearest-point search with the reference's cache semantics (coordinate_converter.py:185-339)."""

    WINDOW = 10.0        # half width of the cached local window [m]      (:223-224)
    WINDOW_SAMPLES = 100  # (:225)
    GLOBAL_STEP = 0.1    # (:322)

    def __init__(self, reference_path):
        self.reference_path = reference_path
        # Batched position evaluation for the ~160 points of one search: ONE calc_position call on
        # an array instead of one call per point.  NumPy evaluates array elements independently with
        # the same inner loops (including its vectorised pow), so the values are bit-identical to the
        # reference's point-by-point calls; only the per-call overhead goes (10 ms -> ~1 ms per plan()).
        self._batched = True
        # Paths that expose their coefficient arrays (ours and the reference's CubicSpline2D) get a lean
        # evaluator: the same element-wise NumPy expression as CubicSpline1D.calc_position
        # (a + b dx + c dx**2.0 + d dx**3.0), with the segment search and the powers shared by x and y.
        self._tab = None
        try:
            from .spline import spline_tables
            t = spline_tables(reference_path)
            self._tab = tuple(t[k] for k in ("knots", "xa", "xb", "xc", "xd", "ya", "yb", "yc", "yd"))
            self._knots_list = [float(v) for v in self._tab[0]]
            self._seg_cols = {}
        except Exception:
            self._tab = None

    # -- search --------------------------------------------------------------------------
    def _xy(self, s):
        px, py = self.reference_path.calc_position(s)
        return _f(px), _f(py)

    def _xy_many(self, s_values):
        """Positions of several arc lengths, element for element what _xy gives."""
        if not self._batched:
            pts = [self._xy(s) for s in s_values]
            return [p[0] for p in pts], [p[1] for p in pts]
        sv = np.asarray(s_values, dtype=np.float64).reshape(-1)
        if self._tab is None:
            px, py = self.reference_path.calc_position(sv)
            return np.atleast_1d(px), np.atleast_1d(py)
        knots, xa, xb, xc, xd, ya, yb, yc, yd = self._tab
        inside = (sv >= knots[0]) & (sv <= knots[-1])                 # cubic_spline.py:62
        i = np.searchsorted(knots, sv, side="right") - 1               # cubic_spline.py:162-165
        i = np.minimum(np.maximum(i, 0), knots.shape[0] - 2)
        dx = sv - knots[i]
        dx2, dx3 = dx ** 2.0, dx ** 3.0
        px = xa[i] + xb[i] * dx + xc[i] * dx2 + xd[i] * dx3            # cubic_spline.py:73-74
        py = ya[i] + yb[i] * dx + yc[i] * dx2 + yd[i] * dx3
        if not inside.all():
            px = np.where(inside, px, np.nan)
            py = np.where(inside, py, np.nan)
        return px, py

    def _xy3(self, s_lo, s_hi, s_mid):
        """Positions of the three points of one refinement step.  They almost always share a spline segment; then
        the segment search is done once on Python floats and x and y are evaluated together as one [2, 3] array
        expression with the segment's coefficients as [2, 1] columns -- the same element-wise NumPy operations
        (subtract, power, multiply, add, in the same order) as `_xy_many`, a third of the calls."""
        tab = self._tab
        if tab is not None and self._batched:
            knots = self._knots_list
            lo, hi = min(s_lo, s_hi, s_mid), max(s_lo, s_hi, s_mid)
            if knots[0] <= lo and hi <= knots[-1]:
                i = min(max(bisect.bisect_right(knots, lo) - 1, 0), len(knots) - 2)      # searchsorted(side="right") - 1, clipped
                if min(max(bisect.bisect_right(knots, hi) - 1, 0), len(knots) - 2) == i:
                    col = self._seg_cols.get(i)
                    if col is None:
                        _, xa, xb, xc, xd, ya, yb, yc, yd = tab
                        col = self._seg_cols[i] = tuple(np.array([[u[i]], [v[i]]]) for u, v in ((xa, ya), (xb, yb), (xc, yc), (xd, yd)))
                    a, b, c, d = col
                    dx = np.array([s_lo, s_hi, s_mid], dtype=np.float64) - tab[0][i]
                    p = a + b * dx + c * dx ** 2.0 + d * dx ** 3.0
                    return p[0], p[1]
        return self._xy_many([s_lo, s_hi, s_mid])

    def _heading_curvature(self, rs):
        """yaw, curvature, curvature rate at rs: CubicSpline2D.calc_yaw / calc_curvature /
        calc_curvature_rate (cubic_spline.py:228-288) with the segment search done once.  The
        derivatives are one-element array expressions and the combinations scalar expressions,
        exactly as those methods evaluate them for a scalar argument."""
        if self._tab is None:
            return (_f(self.reference_path.calc_yaw(rs)), _f(self.reference_path.calc_curvature(rs)),
                    _f(self.reference_path.calc_curvature_rate(rs)))
        knots, xa, xb, xc, xd, ya, yb, yc, yd = self._tab
        sv = np.atleast_1d(np.asarray(rs, dtype=np.float64))
        if not ((sv >= knots[0]) & (sv <= knots[-1])).all():
            return np.nan, np.nan, np.nan
        i = np.searchsorted(knots, sv, side="right") - 1
        i = np.minimum(np.maximum(i, 0), knots.shape[0] - 2)
        h = sv - knots[i]
        h2 = h ** 2.0
        dx = (xb[i] + 2.0 * xc[i] * h + 3.0 * xd[i] * h2)[0]          # cubic_spline.py:100
        dy = (yb[i] + 2.0 * yc[i] * h + 3.0 * yd[i] * h2)[0]
        ddx = (2.0 * xc[i] + 6.0 * xd[i] * h)[0]                       # cubic_spline.py:125
        ddy = (2.0 * yc[i] + 6.0 * yd[i] * h)[0]
        dddx = (6.0 * xd[i])[0]                                        # cubic_spline.py:149
        dddy = (6.0 * yd[i])[0]
        yaw = np.arctan2(dy, dx)                                       # :287
        kappa = (ddy * dx - ddx * dy) / ((dx ** 2 + dy ** 2) ** (3 / 2))   # :246
        a = dx * ddy - dy * ddx
        b = dx * dddy - dy * dddx
        c = dx * ddx + dy * ddy
        d = dx * dx + dy * dy
        return yaw, kappa, b / d ** 1.5 - 3.0 * a * c / d ** 2.5      # :273

    def _global_search(self, x, y):
        length = self.reference_path.s[-1]
        n = max(100, int(length / self.GLOBAL_STEP))
        grid = np.linspace(0, length, n)
        px, py = self.reference_path.calc_position(grid)
        return grid[np.argmin(np.hypot(x - px, y - py))]

    def find_nearest_point_on_path(self, x, y):
        path_end = self.reference_path.s[-1]
        best_s = 0.0
        if hasattr(self, "_prev_s"):
            lo = max(0.0, self._prev_s - self.WINDOW)
            hi = min(path_end, self._prev_s + self.WINDOW)
            nearest = float("inf")
            grid = np.linspace(lo, hi, self.WINDOW_SAMPLES)
            gx, gy = self._xy_many(grid)
            for s, px, py in zip(grid, gx, gy):
                gap = math.hypot(x - px, y - py)
                if gap < nearest:
                    nearest, best_s = gap, s
            # a minimum on the window edge (not the path end) means the cache is stale (:241-248)
            stale = (abs(best_s - lo) < 1e-3 and lo > 0) or (abs(best_s - hi) < 1e-3 and hi < path_end)
            if stale:
                best_s = self._global_search(x, y)
        else:
            best_s = self._global_search(x, y)

        step = 0.2                                   # 20 three-point refinements (:253-280)
        for _ in range(20):
            s_lo = max(0, best_s - step)
            s_hi = min(path_end, best_s + step)
            px3, py3 = self._xy3(s_lo, s_hi, best_s)
            gap_lo = math.hypot(x - px3[0], y - py3[0])
            gap_hi = math.hypot(x - px3[1], y - py3[1])
            gap_c = math.hypot(x - px3[2], y - py3[2])
            if gap_lo < gap_c and gap_lo < gap_hi:
                best_s = s_lo
            elif gap_hi < gap_c and gap_hi < gap_lo:
                best_s = s_hi
            else:
                step *= 0.5
        self._prev_s = best_s

        rs = best_s
        rx, ry = self._xy(rs)
        if np.any(np.isnan([rx, ry])):
            rs = self._global_search(x, y)
            rx, ry = self._xy(rs)
            if np.any(np.isnan([rx, ry])):
                raise ValueError(f"Failed to find valid reference point for position ({x:.2f}, {y:.2f})")
        rtheta, rkappa, rdkappa = self._heading_curvature(rs)
        if np.any(np.isnan([rtheta, rkappa, rdkappa])):
            raise ValueError(f"Failed to calculate reference path properties at s={rs:.2f}")
        return rs, rx, ry, rtheta, rkappa, rdkappa

    # -- formulas ------------------------------------------------------------------------
    @staticmethod
    def cartesian_to_frenet(rs, rx, ry, rtheta, rkappa, rdkappa, x, y, v, a, theta, kappa
                            ) -> Tuple[Tuple[float, float, float], Tuple[float, float, float]]:
        """Apollo-style conversion; returns (s, s', s''), (d, d', d'') with d', d'' SPATIAL
        derivatives (coordinate_converter.py:58-88)."""
        off_x = x - rx
        off_y = y - ry
        cos_r = np.cos(rtheta)
        sin_r = np.sin(rtheta)
        side = cos_r * off_y - sin_r * off_x
        d = np.copysign(np.hypot(off_x, off_y), side)
        delta = theta - rtheta
        tan_delta = np.tan(delta)
        cos_delta = np.cos(delta)
        one_minus_kd = 1 - rkappa * d
        d_prime = one_minus_kd * tan_delta
        kd_prime = rdkappa * d + rkappa * d_prime
        d_pprime = (-kd_prime * tan_delta +
                    one_minus_kd / (cos_delta * cos_delta) * (kappa * one_minus_kd / cos_delta - rkappa))
        s_dot = v * cos_delta / one_minus_kd
        delta_prime = one_minus_kd / cos_delta * kappa - rkappa
        s_ddot = (a * cos_delta - s_dot * s_dot * (d_prime * delta_prime - kd_prime)) / one_minus_kd
        return (rs, s_dot, s_ddot), (d, d_prime, d_pprime)


class BatchCoordinateConverter:
    """Nearest-point search for N independent converters at once (one `_prev_s` cache each).

    The closed-loop driver asks for the nearest path point of every simulation twice per step; done one
    simulation at a time that search is ~95 % of a lock-step.  Here the ~160 path evaluations per search
    are laid out as [N, .] arrays.  Results are bit-identical to N scalar `CoordinateConverter`s:
      * positions are element-wise NumPy expressions (the same inner loops whatever the array length);
      * the distances that only DECIDE (argmin over the window, the three-point refinement) are np.hypot
        here and math.hypot in the reference -- both within an ulp of the true value -- so a decision can
        only differ when two distances of different points lie within a few ulp of each other; those rows
        are recomputed with math.hypot, the reference's own arithmetic, before deciding;
      * everything that enters the returned numbers through libm (atan2, pow, cos, tan) stays a per-query
        scalar expression (`CoordinateConverter._heading_curvature`, `cartesian_to_frenet`).
    """

    NEAR = 16.0 * np.finfo(np.float64).eps

    def __init__(self, reference_path, n: int, engine=None):
        """engine: a SweepEngine built on the same path.  With it, `nearest_s` runs the search on the device
        (fot_nearest_s_device) and recomputes here only the rows whose every decision the device could not certify
        (DESIGN.md section 4e); the results and caches are the same either way.  `device_rows` / `host_rows` count
        the rows each side answered."""
        self.one = CoordinateConverter(reference_path)
        self.path_end = float(reference_path.s[-1])
        self.prev_s = np.full(n, np.nan)
        self._global = None
        self.engine = engine
        self.device_rows = 0
        self.host_rows = 0

    # positions as [rows, cols] arrays
    def _xy_grid(self, s):
        px, py = self.one._xy_many(s.reshape(-1))
        return np.asarray(px).reshape(s.shape), np.asarray(py).reshape(s.shape)

    def _global_search(self, x, y):
        """coordinate_converter.py:319-339 (already array arithmetic in the reference); the grid positions
        do not depend on the query and are computed once."""
        if self._global is None:
            n = max(100, int(self.path_end / CoordinateConverter.GLOBAL_STEP))
            grid = np.linspace(0, self.one.reference_path.s[-1], n)
            px, py = self.one.reference_path.calc_position(grid)
            self._global = (grid, px, py)
        grid, px, py = self._global
        return grid[np.argmin(np.hypot(x - px, y - py))]

    def nearest_s(self, idx, x, y):
        """best_s of find_nearest_point_on_path (coordinate_converter.py:202-283) for converters `idx` at
        the points (x, y); updates their caches."""
        if self.engine is None:
            return self._nearest_s_host(idx, x, y)
        idx = np.asarray(idx, dtype=np.int64)
        x = np.asarray(x, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64)
        best, status = self.engine.nearest_s(x, y, self.prev_s[idx])
        sure = status == 0
        self.prev_s[idx[sure]] = best[sure]
        redo = np.nonzero(~sure)[0]
        if len(redo):                                     # their caches still hold the values from before this call
            best[redo] = self._nearest_s_host(idx[redo], x[redo], y[redo])
        self.device_rows += len(idx) - len(redo)
        self.host_rows += len(redo)
        return best

    def _nearest_s_host(self, idx, x, y):
        idx = np.asarray(idx, dtype=np.int64)
        x = np.asarray(x, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64)
        m = len(idx)
        end = self.path_end
        best = np.zeros(m)
        prev = self.prev_s[idx]
        cached = ~np.isnan(prev)
        rows = np.nonzero(cached)[0]
        if len(rows):
            lo = np.maximum(0.0, prev[rows] - CoordinateConverter.WINDOW)
            hi = np.minimum(end, prev[rows] + CoordinateConverter.WINDOW)
            n_w = CoordinateConverter.WINDOW_SAMPLES
            step = (hi - lo) / (n_w - 1)                                  # np.linspace: k * step + start, last = stop
            grid = np.arange(0, n_w)[None, :] * step[:, None] + lo[:, None]
            grid[:, -1] = hi
            flat = step == 0
            if flat.any():                                                # np.linspace's other branch (k / div * delta)
                for r in np.nonzero(flat)[0]:
                    grid[r] = np.linspace(lo[r], hi[r], n_w)
            px, py = self._xy_grid(grid)
            dist = np.hypot(x[rows, None] - px, y[rows, None] - py)
            two = np.partition(dist, 1, axis=1)[:, :2]
            redo = ~(two[:, 1] - two[:, 0] > self.NEAR * two[:, 1])       # near tie, or a NaN in the row
            for r in np.nonzero(redo)[0]:
                xr, yr = x[rows[r]], y[rows[r]]
                for k in range(n_w):
                    dist[r, k] = math.hypot(xr - px[r, k], yr - py[r, k])
            nan_rows = np.isnan(dist).any(axis=1)
            pick = np.argmin(np.where(np.isnan(dist), np.inf, dist), axis=1)      # `dist < min_dist` skips NaN, first minimum wins
            b = grid[np.arange(len(rows)), pick]
            b = np.where(nan_rows & np.isnan(dist).all(axis=1), 0.0, b)
            stale = ((np.abs(b - lo) < 1e-3) & (lo > 0)) | ((np.abs(b - hi) < 1e-3) & (hi < end))
            for r in np.nonzero(stale)[0]:
                b[r] = self._global_search(x[rows[r]], y[rows[r]])
            best[rows] = b
        for r in np.nonzero(~cached)[0]:
            best[r] = self._global_search(x[r], y[r])

        step = np.full(m, 0.2)
        for _ in range(20):
            s_lo = np.maximum(0.0, best - step)
            s_hi = np.minimum(end, best + step)
            px, py = self._xy_grid(np.stack([s_lo, s_hi, best]))
            g = np.hypot(x[None, :] - px, y[None, :] - py)
            near = lambda a, b_, sa, sb: (np.abs(g[a] - g[b_]) <= self.NEAR * np.maximum(g[a], g[b_])) & (sa != sb)
            redo = near(0, 2, s_lo, best) | near(1, 2, s_hi, best) | near(0, 1, s_lo, s_hi) | np.isnan(g).any(axis=0)
            for r in np.nonzero(redo)[0]:
                for k in range(3):
                    g[k, r] = math.hypot(x[r] - px[k, r], y[r] - py[k, r])
            go_lo = (g[0] < g[2]) & (g[0] < g[1])
            go_hi = ~go_lo & (g[1] < g[2]) & (g[1] < g[0])
            best = np.where(go_lo, s_lo, np.where(go_hi, s_hi, best))
            step = np.where(go_lo | go_hi, step, step * 0.5)
        self.prev_s[idx] = best
        return best

    def reference_points(self, idx, x, y):
        """find_nearest_point_on_path for converters `idx`: arrays rs, rx, ry, rtheta, rkappa, rdkappa and
        `valid` (False where the reference raises)."""
        x = np.asarray(x, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64)
        return self._points_at(self.nearest_s(idx, x, y), x, y)

    def _points_at(self, rs, x, y):
        """The rest of `reference_points` once the nearest arc lengths rs of the points (x, y) are known."""
        rx, ry = (np.array(v, dtype=np.float64) for v in self.one._xy_many(rs))
        valid = np.ones(len(rs), dtype=bool)
        for r in np.nonzero(np.isnan(rx) | np.isnan(ry))[0]:              # coordinate_converter.py:289-296
            rs[r] = self._global_search(x[r], y[r])
            rx[r], ry[r] = self.one._xy(rs[r])
            valid[r] = not (np.isnan(rx[r]) or np.isnan(ry[r]))
        rtheta, rkappa, rdkappa = self._heading_curvature_many(rs)
        valid &= ~(np.isnan(rtheta) | np.isnan(rkappa) | np.isnan(rdkappa))   # :303-307
        return rs, rx, ry, rtheta, rkappa, rdkappa, valid

    def _heading_curvature_many(self, rs):
        """CoordinateConverter._heading_curvature for an array of arc lengths.  The derivative polynomials
        and arctan2 are array expressions there too; the powers are np.float64 SCALAR powers in the reference
        (libm pow, not NumPy's array pow and not a multiplication), hence `_pow`."""
        if self.one._tab is None:
            out = np.array([self.one._heading_curvature(v) for v in rs], dtype=np.float64).reshape(-1, 3)
            return out[:, 0], out[:, 1], out[:, 2]
        knots, xa, xb, xc, xd, ya, yb, yc, yd = self.one._tab
        sv = np.asarray(rs, dtype=np.float64)
        inside = (sv >= knots[0]) & (sv <= knots[-1])
        i = np.searchsorted(knots, sv, side="right") - 1
        i = np.minimum(np.maximum(i, 0), knots.shape[0] - 2)
        h = sv - knots[i]
        h2 = h ** 2.0
        dx = xb[i] + 2.0 * xc[i] * h + 3.0 * xd[i] * h2
        dy = yb[i] + 2.0 * yc[i] * h + 3.0 * yd[i] * h2
        ddx = 2.0 * xc[i] + 6.0 * xd[i] * h
        ddy = 2.0 * yc[i] + 6.0 * yd[i] * h
        dddx = 6.0 * xd[i]
        dddy = 6.0 * yd[i]
        with np.errstate(all="ignore"):
            yaw = np.arctan2(dy, dx)
            kappa = (ddy * dx - ddx * dy) / _pow(_pow(dx, 2.0) + _pow(dy, 2.0), 3 / 2)
            a = dx * ddy - dy * ddx
            b = dx * dddy - dy * dddx
            c = dx * ddx + dy * ddy
            d = dx * dx + dy * dy
            rate = b / _pow(d, 1.5) - 3.0 * a * c / _pow(d, 2.5)
        nan = np.where(inside, 0.0, np.nan)
        return yaw + nan, kappa + nan, rate + nan


class RoutedCoordinateConverter:
    """`BatchCoordinateConverter` for rows on different reference paths: row q searches `paths[route[q]]`.  One device
    search covers every row whatever its route (the engine's routes must be `paths`, in order); the rows it cannot
    certify, and the rest of the conversion, go through the converter of their own route.  Caches, results and the
    device_rows / host_rows counts are those of one BatchCoordinateConverter per route."""

    def __init__(self, paths, route, engine=None):
        from .engine import route_array
        r = np.asarray(route)
        if r.ndim != 1:
            raise ValueError(f"route must be [n], got {list(r.shape)}")
        self.route = route_array(r, len(r), len(paths)).astype(np.int64)     # integers in [0, len(paths)), else ValueError
        n = len(self.route)
        self.parts = [BatchCoordinateConverter(p, n) for p in paths]
        self.prev_s = np.full(n, np.nan)
        for part in self.parts:                            # one cache: row q is only ever touched by its own route's part
            part.prev_s = self.prev_s
        self.engine = engine
        self.device_rows = 0
        self.host_rows = 0

    def _by_route(self, idx):
        """(route, positions in idx of its rows) for every route that idx touches."""
        r = self.route[idx]
        return [(k, np.nonzero(r == k)[0]) for k in np.unique(r)]

    def nearest_s(self, idx, x, y):
        idx = np.asarray(idx, dtype=np.int64)
        x = np.asarray(x, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64)
        best = np.zeros(len(idx))
        if self.engine is None:
            for k, sel in self._by_route(idx):
                best[sel] = self.parts[k]._nearest_s_host(idx[sel], x[sel], y[sel])
            return best
        best, status = self.engine.nearest_s(x, y, self.prev_s[idx], route=self.route[idx])
        sure = status == 0
        self.prev_s[idx[sure]] = best[sure]
        redo = np.nonzero(~sure)[0]
        for k, sel in self._by_route(idx[redo]):          # their caches still hold the values from before this call
            rows = redo[sel]
            best[rows] = self.parts[k]._nearest_s_host(idx[rows], x[rows], y[rows])
        self.device_rows += len(idx) - len(redo)
        self.host_rows += len(redo)
        return best

    def reference_points(self, idx, x, y):
        """BatchCoordinateConverter.reference_points, each row on its own route."""
        idx = np.asarray(idx, dtype=np.int64)
        x = np.asarray(x, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64)
        rs = self.nearest_s(idx, x, y)
        out = [np.empty(len(idx)) for _ in range(6)] + [np.zeros(len(idx), dtype=bool)]
        for k, sel in self._by_route(idx):
            for a, v in zip(out, self.parts[k]._points_at(rs[sel], x[sel], y[sel])):
                a[sel] = v
        return tuple(out)


def _pow(base, exponent: float):
    """np.float64 scalar `**` (libm pow through NumPy's scalar math) for every element of `base`."""
    out = np.empty(len(base))
    for k, v in enumerate(base.tolist()):
        try:
            out[k] = math.pow(v, exponent)
        except (OverflowError, ValueError):
            with np.errstate(all="ignore"):
                out[k] = np.float64(v) ** exponent
    return out


def ego_to_frenet_many(converter: BatchCoordinateConverter, idx, ego, last_kappa):
    """`ego_to_frenet` for converters `idx`: ego [m, 5] (x, y, yaw, v, a), last_kappa [m].  Returns
    (frenet [m, 6], ok [m]); ok False where the reference's plan() returns None.  The conversion formulas
    (coordinate_converter.py:58-88) are ufunc calls and IEEE arithmetic on scalars in the reference; as array
    expressions they give the same element values (tests/test_batch_converter.py)."""
    ego = np.asarray(ego, dtype=np.float64).reshape(-1, 5)
    x, y, theta, v, a = (ego[:, k] for k in range(5))
    kappa = np.asarray(last_kappa, dtype=np.float64)
    rs, rx, ry, rtheta, rkappa, rdkappa, ok = converter.reference_points(idx, x, y)
    with np.errstate(all="ignore"):
        (s, s_d, s_dd), (d, d_p, d_pp) = CoordinateConverter.cartesian_to_frenet(rs, rx, ry, rtheta, rkappa, rdkappa,
                                                                                 x, y, v, a, theta, kappa)
        frenet = np.stack([s, s_d, s_dd, d, d_p * s_d, d_pp * _pow(s_d, 2.0) + d_p * s_dd], axis=1)
    frenet[~ok] = 0.0
    return frenet, ok


def ego_to_frenet(converter: CoordinateConverter, ego_state, last_kappa: float) -> Optional[np.ndarray]:
    """frenet_planner.py:334-374.  Returns [s, s_d, s_dd, d, d_d, d_dd] (time derivatives) or
    None when the conversion fails (the reference logs and returns None)."""
    try:
        ref = converter.find_nearest_point_on_path(ego_state.x, ego_state.y)
        (s, s_d, s_dd), (d, d_p, d_pp) = converter.cartesian_to_frenet(
            *ref, ego_state.x, ego_state.y, ego_state.v, ego_state.a, ego_state.yaw, last_kappa)
        d_d = d_p * s_d
        d_dd = d_pp * s_d ** 2 + d_p * s_dd
        return np.array([s, s_d, s_dd, d, d_d, d_dd], dtype=np.float64)
    except Exception:
        return None
