"""Collision decisions at the collision radius: obstacles a hair inside and outside it, on every sweep path.

Both sweep kernels decide a collision by `dx*dx + dy*dy <= r^2` (fp.py:1196-1198, :1231-1233), but only for the
obstacles that conservative screens let through first: the fp32 trajectory boxes (fot_prepass, box_staged), the box of
the reference points padded by the road width or |d0| plus the collision reach, the tangent-frame window (collision
radius, footprint reach and a 1e-9 slack along the tangent; the clean candidates' lateral range across it), the chunked
obstacle list and the survivor queue, and the clamped time index.  A screen may pass extra obstacles; it must never
drop one the exact test accepts.  Random obstacle fields almost never come within 1e-6 of the radius, so these tests
build the boundary on purpose.  From the oracle's own candidate positions they place an obstacle at r(1 - delta) or
r(1 + delta) from one sample of one candidate, chosen where a screen is tight, and the oracle certifies that exactly
this flips that candidate between COLLISION and another category (the CPU test).  Every batch of such queries then
runs through every sweep path and must give the oracle's categories, costs, winners and histograms (the GPU test).
"""
from __future__ import annotations

import functools
import math
from dataclasses import dataclass, field
from typing import Optional

import numpy as np
import pytest

from oracle import frenet_oracle as O
from tests import runners, scenarios

# 5 horizons x 3 terminal speeds x 7 lateral targets + 9 brake horizons = 114 candidates: ~25 ms per oracle call
K_SMALL = dict(scenarios.S1_KNOBS, d_road_w=0.9, d_t_s=3.0, min_t=4.6)
DELTAS = (1e-10, 1e-8, 1e-6)
FAR_DELTAS = (1e-6, 1e-4)            # far from the origin positions carry ~1e-9 m of rounding
FAR = np.array([700.0, 900.0])       # offset of "far away": beyond every trajectory and every padded box
FAR_ORIGIN = (3.5e5, 5.6e6)


@dataclass
class Setup:
    knobs: dict
    wp: tuple
    fs: tuple
    targets: tuple                   # names of the (candidate, sample) picks, see `pick`
    target_speed: float = 6.0
    t_obs: int = 0                   # obstacle horizon; 0: the time grid's length
    footprint: Optional[tuple] = None
    dist_s: int = 0                  # samples of a distribution; 0: single-sample mode
    deltas: tuple = DELTAS
    extra: tuple = ()                # further case families: "inflation", "nan_inf", "crowd"


def _shift(wp, dx, dy):
    return ([x + dx for x in wp[0]], [y + dy for y in wp[1]])


MAIN = ("lat_first", "lat_last", "s31", "s32", "s33", "last", "brake_hold")
SETUPS = {
    "straight": Setup(K_SMALL, scenarios.STRAIGHT_60, (5.0, 5.0, 0.0, 0.3, 0.0, 0.0), MAIN, extra=("nan_inf",)),
    "s_curve": Setup(K_SMALL, scenarios.s_curve_waypoints(), (10.0, 5.0, 0.0, 0.2, 0.0, 0.0), MAIN),
    "arc": Setup(K_SMALL, scenarios.arc_waypoints(), (3.0, 4.0, 0.0, 0.1, 0.0, 0.0), ("lat_first", "lat_last", "s32", "last", "brake_hold")),
    # |d0| = 2.9 > max_road_width = 2.7: sample 0 lies outside the road, where only the |d0| term of the pad reaches
    "off_road_start": Setup(K_SMALL, scenarios.STRAIGHT_60, (5.0, 5.0, 0.0, 2.9, -2.0, 0.0), ("start_first", "start_second")),
    "spline_end": Setup(K_SMALL, scenarios.STRAIGHT_60, (40.0, 5.0, 0.0, -0.3, 0.0, 0.0), ("trunc_last", "trunc_last_b")),
    "short_horizon": Setup(K_SMALL, scenarios.STRAIGHT_60, (5.0, 5.0, 0.0, 0.3, 0.0, 0.0), ("past_t_obs",), t_obs=30),
    "inflation_1.3": Setup(dict(K_SMALL, collision_margin_inflation=1.3), scenarios.s_curve_waypoints(),
                           (10.0, 5.0, 0.0, 0.2, 0.0, 0.0), (), extra=("inflation",)),
    "inflation_0.8": Setup(dict(K_SMALL, collision_margin_inflation=0.8), scenarios.STRAIGHT_60,
                           (5.0, 5.0, 0.0, 0.3, 0.0, 0.0), (), extra=("inflation",)),
    "footprint": Setup(K_SMALL, scenarios.s_curve_waypoints(), (10.0, 5.0, 0.0, 0.2, 0.0, 0.0),
                       ("rear_circle", "mid_circle", "front_circle"), footprint=(4.5, 2.0, 3)),
    # chance_epsilon 0.25 of 8 samples: a candidate may violate in floor(2.0) = 2 samples
    "distribution": Setup(dict(K_SMALL, chance_epsilon=0.25), scenarios.arc_waypoints(), (3.0, 4.0, 0.0, 0.1, 0.0, 0.0),
                          ("lat_last", "s32", "brake_hold"), dist_s=8),
    "crowd": Setup(K_SMALL, scenarios.s_curve_waypoints(), (10.0, 5.0, 0.0, 0.2, 0.0, 0.0), (), extra=("crowd",)),
    # 129 samples per candidate: beyond fot_sweep_pairs, so fot_sweep_items runs on every path
    "long_grid": Setup(dict(K_SMALL, dt=0.05, min_t=6.0, max_t=6.4), scenarios.STRAIGHT_60, (5.0, 5.0, 0.0, 0.3, 0.0, 0.0),
                       ("lat_last", "s100", "last", "brake_hold")),
    # the window subtracts products of ~5.6e6 here
    "far_from_origin": Setup(K_SMALL, _shift(scenarios.s_curve_waypoints(), *FAR_ORIGIN), (10.0, 5.0, 0.0, 0.2, 0.0, 0.0),
                             ("lat_first", "lat_last", "s32", "last", "brake_hold"), deltas=FAR_DELTAS),
}


# ---------------------------------------------------------------------------------------------
# construction (oracle only)
# ---------------------------------------------------------------------------------------------
def oracle_planner(s: Setup) -> O.OraclePlanner:
    kn = O.Knobs(**s.knobs)
    fp = runners.make_footprint(s.footprint)
    if fp is not None:
        kn.footprint_offsets, kn.footprint_radius = fp.offsets, fp.radius
    return O.OraclePlanner(O.Spline2D(*s.wp), kn)


def radii(s: Setup):
    """(static radius, dynamic radius) as collision_geometry has them (fp.py:1172-1175): the inflation applies to
    single-sample dynamic obstacles only."""
    ego = runners.make_footprint(s.footprint).radius if s.footprint else s.knobs["robot_radius"]
    r = max(ego + s.knobs["obstacle_radius"], 1e-6)
    return r, (r if s.dist_s else r * s.knobs.get("collision_margin_inflation", 1.0))


def n_total(s: Setup) -> int:
    return int(round(s.knobs["max_t"] / s.knobs["dt"])) + 1


def t_obs(s: Setup) -> int:
    return s.t_obs or n_total(s)


@functools.lru_cache(maxsize=None)
def base(name):
    """The obstacle-free oracle run of a setup: (result, candidates)."""
    s = SETUPS[name]
    pl = oracle_planner(s)
    res = pl.plan_frenet(s.fs, np.empty((0, 2)), None, s.target_speed)
    return res, pl.last_candidates


@dataclass(frozen=True)
class Target:
    name: str
    cand: int
    n: int
    circle: Optional[int] = None     # footprint circle the obstacle is placed at


def pick(name, which) -> Target:
    """(candidate, sample) of the setup where the screen `which` is tight; the candidate is OK without obstacles."""
    s = SETUPS[name]
    res, cands = base(name)
    kn = O.Knobs(**s.knobs)
    n_d, n_grid = len(O.lateral_grid(kn)), len(O.horizon_grid(kn)) * len(O.speed_grid(kn, s.target_speed))
    ok = [i for i, c in enumerate(cands) if c.category == O.CAT_OK]
    full = [i for i in ok if i < n_grid * n_d and cands[i].keep == n_total(s)]      # longest horizon, untruncated
    mid = [i for i in full if i % n_d == n_d // 2]
    if which in ("lat_first", "lat_last"):
        # the edge of the lateral grid, late in the horizon: the window's d_lo / d_hi come from the grid ends
        i = [i for i in full if i % n_d == (0 if which == "lat_first" else n_d - 1)][0]
        return Target(which, i, int(0.8 * (n_total(s) - 1)))
    if which in ("s31", "s32", "s33", "s100"):
        return Target(which, mid[0], int(which[1:]))                 # around the pair kernel's 32-sample passes
    if which == "last":
        return Target(which, mid[0], cands[mid[0]].keep - 1)
    if which == "brake_hold":
        # a brake-ladder candidate in its held tail: samples past the brake horizon repeat its end state
        i = [i for i in ok if i >= n_grid * n_d][0]
        hold = int(round(O.brake_horizons(kn)[i - n_grid * n_d] / kn.dt))
        n = (hold + n_total(s) - 1) // 2 + 1
        assert hold < n < cands[i].keep
        return Target(which, i, n)
    if which in ("start_first", "start_second"):
        return Target(which, ok[0 if which == "start_first" else -1], 0)
    if which in ("trunc_last", "trunc_last_b"):
        i = [i for i in ok if cands[i].keep < res.n_points[i]][0 if which == "trunc_last" else -1]
        return Target(which, i, cands[i].keep - 1)                  # the last kept sample of a candidate cut at the spline end
    if which == "past_t_obs":
        return Target(which, mid[0], t_obs(s) + 10)                 # clamps to obstacle step T_obs - 1
    if which in ("rear_circle", "mid_circle", "front_circle"):
        return Target(which, mid[0], 32, ("rear_circle", "mid_circle", "front_circle").index(which))
    raise KeyError(which)


def anchor(s: Setup, t: Target):
    """(point, unit heading) the obstacle is placed around: the candidate's position at sample n, or the centre of its
    footprint circle there."""
    c = base_cands(s)[t.cand]
    h = np.array([np.cos(c.yaw[t.n]), np.sin(c.yaw[t.n])])
    p = np.array([c.x[t.n], c.y[t.n]])
    if t.circle is not None:
        p = p + runners.make_footprint(s.footprint).offsets[t.circle] * h
    return p, h


def base_cands(s: Setup):
    return base(next(k for k, v in SETUPS.items() if v is s))[1]


def direction(which, h):
    nrm = np.array([-h[1], h[0]])
    return {"head": h, "back": -h, "across": nrm, "across-": -nrm, "diag": (h + nrm) / math.sqrt(2.0),
            "+x": np.array([1.0, 0.0]), "-x": np.array([-1.0, 0.0]), "+y": np.array([0.0, 1.0]),
            "-y": np.array([0.0, -1.0])}[which]


def place(s: Setup, t: Target, radius, delta, inside, which):
    p, h = anchor(s, t)
    return p + radius * (1.0 - delta if inside else 1.0 + delta) * direction(which, h)


def blink(s: Setup, t: Target, o):
    """A predicted trajectory that is far away except at the time step sample t.n is tested against."""
    tr = np.tile(anchor(s, t)[0] + FAR, (t_obs(s), 1))
    tr[min(t.n, t_obs(s) - 1)] = o
    return tr


def still(s: Setup, o):
    """A predicted trajectory that stands at o: its box is one point."""
    return np.tile(o, (t_obs(s), 1))


def still_side(s: Setup, t: Target, radius, prefer):
    """The side (across / across-) from which an obstacle standing still, or a static point, is nearer to the target
    sample than to every other sample and circle of the candidate (on a curve: the outer side)."""
    c = base_cands(s)[t.cand]
    pts = np.stack([c.x, c.y], axis=1)
    if s.footprint:
        h = np.stack([np.cos(c.yaw), np.sin(c.yaw)], axis=1)
        pts = np.concatenate([pts + off * h for off in runners.make_footprint(s.footprint).offsets])
    p = anchor(s, t)[0]
    for side in (prefer, STILL_DIRS[1 - STILL_DIRS.index(prefer)]):
        o = place(s, t, radius, 0.0, False, side)
        others = np.hypot(*(pts - o).T)[np.any(pts != p, axis=1)]     # the held tail of a brake profile repeats p
        if others.min() > radius * (1.0 + 1e-12):
            return side
    raise AssertionError(("no sharp side", t))


# obstacle shapes and directions: a trajectory that stands still is closest to a straight-moving sample from across
# its heading only; one that is near at a single time step can come from anywhere
BLINK_DIRS = ("head", "back", "diag", "+x", "-x", "+y", "-y", "across")
STILL_DIRS = ("across", "across-")


@dataclass
class Case:
    label: str
    target: Target
    hit: bool                        # the oracle must put the target in COLLISION (True) or elsewhere (False)
    dyn: list = field(default_factory=list)      # single-sample: [T, 2] trajectories; distribution: [S, T, 2] each
    static: list = field(default_factory=list)   # [2] points


def make_cases(name):
    """The queries of one setup (one batch), each with the category its construction forces on its target."""
    s = SETUPS[name]
    r, r_dyn = radii(s)
    out = []
    for k, which in enumerate(s.targets):
        t = pick(name, which)
        for j, delta in enumerate(s.deltas):
            for inside in (True, False):
                tag = f"{which} d={delta:g} {'in' if inside else 'out'}"
                if s.dist_s:
                    # exactly `allowed` violating samples, then one more (fp.py:1113-1124)
                    allowed = int(math.floor(s.knobs["chance_epsilon"] * s.dist_s))
                    bad = allowed + (0 if inside else 1)
                    d = BLINK_DIRS[(k + j) % len(BLINK_DIRS)]
                    samples = [blink(s, t, place(s, t, r, delta, m < bad, d)) for m in range(s.dist_s)]
                    out.append(Case(f"{tag}: {bad} of {s.dist_s} samples inside, {d}", t, bad > allowed, dyn=[np.stack(samples)]))
                    continue
                if t.circle is not None:
                    dirs = ["across", "across-"] + (["back"] if t.circle == 0 else ["head"] if t.circle == 2 else [])
                    for d in dirs:
                        out.append(Case(f"{tag} blink {d}", t, inside, dyn=[blink(s, t, place(s, t, r_dyn, delta, inside, d))]))
                    side = still_side(s, t, r, "across")
                    out.append(Case(f"{tag} static {side}", t, inside, static=[place(s, t, r, delta, inside, side)]))
                    continue
                # two blink directions and one standing obstacle per (target, delta, side), rotating through the directions
                dirs = (BLINK_DIRS[(2 * k + j) % len(BLINK_DIRS)], BLINK_DIRS[(2 * k + j + 1) % len(BLINK_DIRS)])
                if t.n >= t_obs(s) - 1:                   # every later sample meets the obstacle's last step too
                    dirs = (still_side(s, t, r_dyn, STILL_DIRS[j % 2]),)
                for d in dirs:
                    out.append(Case(f"{tag} blink {d}", t, inside, dyn=[blink(s, t, place(s, t, r_dyn, delta, inside, d))]))
                d = still_side(s, t, r_dyn, STILL_DIRS[(k + j) % 2])
                out.append(Case(f"{tag} still {d}", t, inside, dyn=[still(s, place(s, t, r_dyn, delta, inside, d))]))
    if "nan_inf" in s.extra:
        t = pick(name, "s32")
        for delta in s.deltas:
            o = place(s, t, r_dyn, delta, True, "diag")
            for j, bad in ((5, [np.nan, 0.0]), (45, [0.0, np.nan]), (0, [np.nan, np.nan])):
                tr = blink(s, t, o)
                tr[j] = bad
                # a NaN anywhere makes np.min / np.max NaN: the prefilter drops the whole trajectory (fp.py:1211-1222)
                out.append(Case(f"nan at step {j}, d={delta:g} in", t, False, dyn=[tr]))
            for inside in (True, False):
                o = place(s, t, r_dyn, delta, inside, "across")
                for j, bad in ((7, [np.inf, 0.0]), (40, [-np.inf, np.inf])):
                    tr = blink(s, t, o)
                    tr[j] = bad
                    # an infinite step only widens the box: the boundary step decides
                    out.append(Case(f"inf at step {j}, d={delta:g} {'in' if inside else 'out'}", t, inside, dyn=[tr]))
    if "inflation" in s.extra:
        # single-sample dynamic at r * inflation, static at r; both kinds in one query
        t = pick(name, "lat_last")
        for delta in s.deltas:
            for inside in (True, False):
                tag = f"d={delta:g} {'in' if inside else 'out'}"
                dyn_o = blink(s, t, place(s, t, r_dyn, delta, inside, "head"))
                st_o = place(s, t, r, delta, inside, still_side(s, t, r, "across"))
                miss_dyn = blink(s, t, place(s, t, r_dyn, 1e-3, False, "head"))
                miss_st = place(s, t, r, 1e-3, False, still_side(s, t, r, "across"))
                out.append(Case(f"dynamic {tag}", t, inside, dyn=[dyn_o]))
                out.append(Case(f"static {tag}", t, inside, static=[st_o]))
                out.append(Case(f"dynamic {tag} + static out", t, inside, dyn=[dyn_o], static=[miss_st]))
                out.append(Case(f"static {tag} + dynamic out", t, inside, dyn=[miss_dyn], static=[st_o]))
    if "crowd" in s.extra:
        # 40 dynamic + 40 static boundary obstacles along one candidate: more than one list chunk (64 entries) and
        # more survivors than the queue holds; one of them (listed late) decides
        t0 = pick(name, "lat_last")
        keep = base(name)[1][t0.cand].keep
        for delta in s.deltas:
            for hit_at in (None, "dyn", "static"):
                dyn, st = [], []
                for m in range(40):
                    t = Target("crowd", t0.cand, 5 + m * (keep - 6) // 40)
                    side = "across" if m % 2 else "across-"
                    dyn.append(blink(s, t, place(s, t, r_dyn, delta, hit_at == "dyn" and m == 37, side)))
                    st.append(place(s, t, r, delta, hit_at == "static" and m == 38, "across-" if m % 2 else "across"))
                out.append(Case(f"crowd d={delta:g} decisive={hit_at}", t0, hit_at is not None, dyn=dyn, static=st))
    return out


def batch(name):
    """The setup's queries as batch arrays: frenet [n_q, 6], obstacle tensor [n_q, S, P, T, 2] (padded with far-away
    trajectories), static points [n_q, M, 2] or None (padded with far-away points)."""
    s = SETUPS[name]
    cases = make_cases(name)
    far = np.array([s.wp[0][0], s.wp[1][0]]) + FAR
    S = max(1, s.dist_s)
    P = max(1, max(len(c.dyn) for c in cases))
    M = max(len(c.static) for c in cases)
    dyn = np.empty((len(cases), S, P, t_obs(s), 2))
    dyn[:] = far
    stat = np.empty((len(cases), M, 2)) if M else None
    for q, c in enumerate(cases):
        for p, tr in enumerate(c.dyn):
            dyn[q, :, p] = tr
        if M:
            stat[q] = far
            if c.static:
                stat[q, :len(c.static)] = c.static
    return np.tile(np.asarray(s.fs, dtype=float), (len(cases), 1)), dyn, stat


@functools.lru_cache(maxsize=None)
def oracle_results(name):
    """The oracle on every query of the batch, exactly as the batch holds it (padding included)."""
    s = SETUPS[name]
    pl = oracle_planner(s)
    frenet, dyn, stat = batch(name)
    out = []
    for q in range(len(frenet)):
        st = np.empty((0, 2)) if stat is None else stat[q]
        if s.dist_s:
            out.append(pl.plan_frenet(tuple(frenet[q]), st, None, s.target_speed, dist=dyn[q]))
        else:
            out.append(pl.plan_frenet(tuple(frenet[q]), st, dyn[q, 0], s.target_speed))
    return out


@pytest.mark.parametrize("name", list(SETUPS))
def test_constructions_flip_their_target_in_the_oracle(name):
    """Every construction decides its target candidate: COLLISION when placed inside, another category outside; and
    the targets are candidates that reach the collision test (OK without obstacles)."""
    res0, cands = base(name)
    cases = make_cases(name)
    refs = oracle_results(name)
    assert len(cases) == len(refs) > 0
    hits = 0
    for c, ref in zip(cases, refs):
        assert res0.categories[c.target.cand] == O.CAT_OK, (name, c.label)
        got = int(ref.categories[c.target.cand])
        assert (got == O.CAT_COLL) == c.hit, (name, c.label, got)
        hits += c.hit
    assert 0 < hits < len(cases)


# ---------------------------------------------------------------------------------------------
# every sweep path against the oracle (GPU)
# ---------------------------------------------------------------------------------------------
PAIR_STATIC, PAIR_FOOTPRINT, PAIR_BUDGET, PAIR_OUTPUTS, PAIR_LOOSE, PAIR_ALL = 1, 2, 4, 8, 16, 31
PAIR_INSTANCES = (0, PAIR_STATIC, PAIR_OUTPUTS, PAIR_STATIC | PAIR_OUTPUTS, PAIR_LOOSE, PAIR_BUDGET,
                  PAIR_STATIC | PAIR_FOOTPRINT, PAIR_ALL)    # fot_api.cu FOT_PAIR_INSTANCES, smallest first
ENV = {"pairs": {}, "pairs_no_candidates": {}, "pairs_every_mode": dict(FOT_PAIR_SIMPLE=0), "items": dict(FOT_SWEEP="items"),
       "unstaged": dict(FOT_STAGE_DYN=0), "items_queue_4": dict(FOT_SWEEP="items", FOT_QCAP=4)}
PATHS = tuple(ENV) + ("resident", "gated")


def expected_features(s: Setup, stat, cands: bool, unstaged: bool, every_mode: bool) -> int:
    """The fot_sweep_pairs instantiation the host must pick for this batch (fot_api.cu: the smallest instantiated
    superset of the modes the batch needs)."""
    if every_mode:
        return PAIR_ALL
    need = (PAIR_STATIC if stat is not None else 0) | (PAIR_FOOTPRINT if s.footprint else 0) | \
        (PAIR_BUDGET if s.dist_s and math.floor(s.knobs.get("chance_epsilon", 0.0) * s.dist_s) > 0 else 0) | \
        (PAIR_OUTPUTS if cands else 0) | (PAIR_LOOSE if unstaged else 0)
    return next(f for f in PAIR_INSTANCES if f & need == need)


@functools.lru_cache(maxsize=1)
def filler(n):
    import bench
    _, frenet, dyn = bench.make_queries(0, n)
    return frenet, dyn[:, 0]


def run_path(pl, s: Setup, path, frenet, dyn, stat):
    """One sweep of the batch on `path`: (SweepResult, rows of the setup's queries, sweep kind, pair features)."""
    import torch
    from integrated_path_planning_b200 import _lib
    from integrated_path_planning_b200.batch import DeviceBatch
    lib, h = pl.engine.lib, pl.engine._h
    kw = dict(distribution=dyn) if s.dist_s else dict(dynamic_obstacles=dyn[:, 0])
    n = len(frenet)
    if path in ENV:
        with runners.fot_env(**ENV[path]):
            res = pl.plan_batch(frenet, s.target_speed, static_obstacles=stat, want_candidates=path != "pairs_no_candidates", **kw)
            return res, np.arange(n), int(lib.fot_last_sweep_kind(h)), int(lib.fot_last_pair_features(h))
    mode = _lib.FOT_DYN_DISTRIBUTION if s.dist_s else _lib.FOT_DYN_SINGLE
    if path == "resident":
        db = DeviceBatch(pl, frenet, s.target_speed, dyn, mode, static_obstacles=stat)
        db.launch()
        torch.cuda.synchronize()
        return db.sweep_result(), np.arange(n), int(lib.fot_last_sweep_kind(h)), int(lib.fot_last_pair_features(h))
    # gated host-pointer call: behind the boundary queries 1024 config-4 queries (pedestrian fields cut or padded to the
    # batch's shape), and far-away trajectories up to an upload of more than 8 MB: above both thresholds the host
    # pointer call cuts the batch into ranges and launches the sweep gated on the upload, so that the sweep boxes the
    # trajectories itself (box_staged)
    f_frenet, f_ped = filler(1024)
    S, P, T = dyn.shape[1:4]
    P_g = max(P, -(-600 // (S * T)))
    far = np.array([s.wp[0][0], s.wp[1][0]]) + FAR
    big = np.empty((n + len(f_frenet), S, P_g, T, 2))
    big[:] = far
    big[:n, :, :P] = dyn
    ped = f_ped[:, :min(P_g, f_ped.shape[1])]
    ped = ped[:, :, np.minimum(np.arange(T), ped.shape[2] - 1)]
    big[n:, :, :ped.shape[1]] = ped[:, None]
    assert len(big) >= 1024 and big[:, :, :, :, 0].size * 16 > (8 << 20)
    st = None if stat is None else np.concatenate([stat, np.broadcast_to(far, (len(f_frenet),) + stat.shape[1:])])
    kw = dict(distribution=big) if s.dist_s else dict(dynamic_obstacles=big[:, 0])
    res = pl.plan_batch(np.concatenate([frenet, f_frenet]), s.target_speed, static_obstacles=st, want_candidates=True, **kw)
    return res, np.arange(n), int(lib.fot_last_sweep_kind(h)), int(lib.fot_last_pair_features(h))


def check(name, path, res, rows, refs, cases):
    for q, ref in zip(rows, refs):
        label = (name, path, cases[q].label)
        if res.cand_cat is not None:
            n_c = len(ref.categories)
            assert int(res.n_cand[q]) == n_c, label
            cats = res.cand_cat[q, :n_c].astype(np.int8)
            bad = np.nonzero(cats != ref.categories)[0]
            assert bad.size == 0, (label, "category", bad[:8], cats[bad[:8]], ref.categories[bad[:8]])
            if res.cand_cost is not None:
                np.testing.assert_allclose(res.cand_cost[q, :n_c], ref.costs, rtol=runners.RTOL, atol=0, err_msg=str(label))
        assert int(res.best_idx[q]) == ref.best_index, (label, int(res.best_idx[q]), ref.best_index)
        if ref.best_index >= 0:
            np.testing.assert_allclose(float(res.best_cost[q]), ref.cost, rtol=runners.RTOL, atol=0, err_msg=str(label))
        want = [ref.stats.get(k, 0) for k in runners.GOLDEN_STAT_KEYS]
        assert res.stats[q].tolist() == want, (label, res.stats[q].tolist(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SETUPS))
def test_boundary_obstacles_on_every_sweep_path(name):
    from integrated_path_planning_b200 import BatchFrenetPlanner, CubicSpline2D
    s = SETUPS[name]
    cases, refs = make_cases(name), oracle_results(name)
    frenet, dyn, stat = batch(name)
    pl = BatchFrenetPlanner(CubicSpline2D(*s.wp), footprint=runners.make_footprint(s.footprint), **s.knobs)
    pairs_fit = pl.engine.n_t_max <= 56
    for path in PATHS:
        res, rows, kind, feat = run_path(pl, s, path, frenet, dyn, stat)
        check(name, path, res, rows, refs, cases)
        if path.startswith("items") or not pairs_fit:
            assert (kind, feat) == (1, -1), (name, path, kind, feat)
        elif path != "gated":
            cands = path not in ("pairs_no_candidates", "resident")
            assert kind == 4 and feat == expected_features(s, stat, cands, path == "unstaged", path == "pairs_every_mode"), \
                (name, path, kind, feat)
        else:
            assert kind in (1, 4), (name, path, kind)
