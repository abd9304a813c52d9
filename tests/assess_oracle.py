"""NumPy restatement of trajectory assessment (fot_assess_trajectories; include/fot.h, DESIGN.md section 4i).

The geometry is the reference's, as oracle/frenet_oracle.py restates it in collision_geometry, hits_static and
hits_dynamic (frenet_planner.py:1126-1233): circle centres (x, y) + offset * (cos yaw, sin yaw), the obstacle time index
clip(round(t / dt), 0, T_obs - 1), squared distances dx*dx + dy*dy, pedestrian trajectories with a NaN anywhere
dropped.  This module only adds what the planner throws away: the minimum and where it is, and the counts."""
from __future__ import annotations

import numpy as np


def _argmin(d2: np.ndarray):
    """(min d2, its multi-index) over the non-NaN entries of d2, first in C order on ties (np.argmin); (inf, None)
    when every entry is NaN or there is none."""
    flat = d2.reshape(-1)
    valid = np.flatnonzero(~np.isnan(flat))
    if valid.size == 0:
        return np.inf, None
    i = int(valid[np.argmin(flat[valid])])
    return float(flat[i]), tuple(int(v) for v in np.unravel_index(i, d2.shape))


def centres(x, y, yaw, offsets=None) -> np.ndarray:
    """[n, n_circ, 2] circle centres of the samples (collision_geometry, frenet_planner.py:1152-1160)."""
    pts = np.stack([np.asarray(x, dtype=float), np.asarray(y, dtype=float)], axis=1)
    if offsets is None or len(offsets) == 0:
        return pts[:, None, :]
    heading = np.stack([np.cos(np.asarray(yaw, dtype=float)), np.sin(np.asarray(yaw, dtype=float))], axis=1)
    off = np.asarray(offsets, dtype=float)
    return pts[:, None, :] + off[None, :, None] * heading[:, None, :]


def assess_trajectory(t, x, y, yaw, dt, static=None, dyn=None, r2=((0.0, 0.0),), offsets=None) -> dict:
    """One trajectory -- samples [0, len(x)) of t, x, y, yaw -- against static points [M, 2] and dynamic obstacles
    [S, P, T_obs, 2], under threshold pairs r2 [n_r, 2] = (r2_dyn, r2_static).  Returns the outputs of the table in
    include/fot.h for this (q, j): dyn_min, dyn_at (n, circle, s, p), static_min, static_at (n, circle, point),
    dyn_hits [n_r], first_hit [n_r], static_hit [n_r]."""
    n = len(x)
    r2 = np.asarray(r2, dtype=float).reshape(-1, 2)
    n_r = r2.shape[0]
    out = {"dyn_min": np.inf, "dyn_at": np.full(4, -1), "static_min": np.inf, "static_at": np.full(3, -1),
           "dyn_hits": np.zeros(n_r, dtype=np.int64), "first_hit": np.full(n_r, -1),
           "static_hit": np.zeros(n_r, dtype=np.int64)}
    if n == 0:
        return out
    pts = centres(x[:n], y[:n], np.asarray(yaw)[:n] if offsets is not None and len(offsets) else None, offsets)
    hit_n = np.zeros((n, n_r), dtype=bool)
    with np.errstate(invalid="ignore", over="ignore"):
        if static is not None and len(static) > 0:
            st = np.asarray(static, dtype=float).reshape(-1, 2)
            diff = pts[:, :, None, :] - st[None, None, :, :]                       # [n, n_circ, M, 2]
            d2 = diff[..., 0] * diff[..., 0] + diff[..., 1] * diff[..., 1]
            m, at = _argmin(d2)
            if at is not None:
                out["static_min"], out["static_at"] = np.sqrt(m), np.array(at)
            h = d2[..., None] <= r2[:, 1]                                          # [n, n_circ, M, n_r]
            out["static_hit"] = h.any(axis=(0, 1, 2)).astype(np.int64)
            hit_n |= h.any(axis=(1, 2))
        if dyn is not None and np.size(dyn) > 0:
            dyn = np.asarray(dyn, dtype=float)
            T = dyn.shape[2]
            keep = ~np.isnan(dyn).any(axis=(2, 3))                                 # [S, P]: the NaN-box rule
            k = np.clip(np.round(np.asarray(t, dtype=float)[:n] / dt).astype(int), 0, T - 1)
            obs = dyn[:, :, k, :].transpose(2, 0, 1, 3)                            # [n, S, P, 2]
            diff = pts[:, :, None, None, :] - obs[:, None]                         # [n, n_circ, S, P, 2]
            d2 = diff[..., 0] * diff[..., 0] + diff[..., 1] * diff[..., 1]
            d2 = np.where(keep[None, None], d2, np.nan)
            m, at = _argmin(d2)
            if at is not None:
                out["dyn_min"], out["dyn_at"] = np.sqrt(m), np.array(at)
            h = d2[..., None] <= r2[:, 0]                                          # [n, n_circ, S, P, n_r]
            out["dyn_hits"] = h.any(axis=(0, 1, 3)).sum(axis=0).astype(np.int64)
            hit_n |= h.any(axis=(1, 2, 3))
    for r in range(n_r):
        if hit_n[:, r].any():
            out["first_hit"][r] = int(np.argmax(hit_n[:, r]))
    return out


def verdict(a: dict, chance_epsilon: float, S: int, distribution: bool) -> bool:
    """Collision-free under threshold pair 0 as the planner decides it (frenet_planner.py:1035-1124)."""
    allowed = int(np.floor(chance_epsilon * S)) if distribution else 0
    return bool(a["static_hit"][0] == 0 and a["dyn_hits"][0] <= allowed)
