"""Batched planning: many independent queries per launch, sharded over GPUs.

A query is one reference `plan()` call (ego Frenet state + obstacle field + per-call knobs).
Queries share only the planner constants, so a batch shards across ranks with no traffic
during compute; `gather_winners` is the single collective (SURVEY.md section 8e).
"""
from __future__ import annotations

import dataclasses
from typing import Optional

import numpy as np

from . import _lib
from .engine import (ASSESS_FIELDS, SweepEngine, SweepResult, assess_radii, fot_batch, fot_result, query_arrays, route_array,
                     winner_fields)
from .frenet_host import BatchCoordinateConverter, RoutedCoordinateConverter, ego_to_frenet_many
from .planner import FrenetPlanner


def shard_bounds(n_q: int, world_size: int, rank: int):
    """Contiguous block of ceil(n_q / world_size) queries for `rank`."""
    per = (n_q + world_size - 1) // world_size
    lo = min(rank * per, n_q)
    return lo, min(lo + per, n_q)


class BatchFrenetPlanner(FrenetPlanner):
    """FrenetPlanner plus `plan_batch` (host arrays, Frenet states), `plan_batch_from_ego` (host arrays, ego states)
    and `plan_batch_device` (torch buffers)."""

    def plan_batch(self, frenet_states, target_speed, dynamic_obstacles=None, distribution=None,
                   static_obstacles=None, constraint_overrides=None, limits=None, max_stop_distance=None,
                   want_candidates: bool = False, winner_samples: int = 0, top_k: int = 0,
                   rank_series: bool = True, cost_weights=None, weight_series: bool = True,
                   cost_terms: bool = False, route=None, assess: bool = False, assess_obstacles=None,
                   assess_r2=None, assess_candidates: bool = False) -> SweepResult:
        """frenet_states [n_q,6]; target_speed scalar or [n_q]; dynamic_obstacles [n_q,P,T,2] or
        distribution [n_q,S,P,T,2]; static_obstacles [M,2] (shared) or [n_q,M,2]; limits [n_q,4]
        overrides constraint_overrides; max_stop_distance scalar / [n_q] (NaN = none); winner_samples = k > 0
        reads back only the first k samples of each winner series (`engine.fetch_winners` for the rest).
        top_k > 0: also the top_k best feasible candidates of every query (`SweepResult.rank_*`, `alternatives`),
        with their series unless rank_series is False.  cost_weights [n_w,6] (every query) or [n_q,n_w,6] (columns
        _lib.COST_WEIGHT_KEYS): also every query's winner under each weighting (`SweepResult.w_*`, `under_weights`),
        with its series unless weight_series is False.  cost_terms: also the five cost terms of every candidate
        (`SweepResult.cost_terms`).  With any of these the batch runs as a device-resident `DeviceBatch`.  route: the
        reference path of every query, an id into `routes` (`add_route`), one for all queries or [n_q]; None: route 0.
        A routed query gives what a planner built on its route gives.  assess: also the closest approach and collision
        counts of the winner (and of the ranked alternatives with top_k > 0) against the batch's own obstacle field, or
        against assess_obstacles [n_q, S, P, T, 2], under the threshold pairs assess_r2 (`DeviceBatch`;
        `SweepResult.assessed`, `assessment`).  assess_candidates: the same assessment for every generated candidate,
        the rejected ones included, against the same field and pairs (`SweepResult.cand_assessed`,
        `candidate_assessment`; with want_candidates the table's categories and costs come along)."""
        q, _ = self._batch_arrays(frenet_states, target_speed, dynamic_obstacles, distribution, static_obstacles,
                                  constraint_overrides, limits, max_stop_distance, route=route)
        return self._run(q, want_candidates, winner_samples, top_k, rank_series, cost_weights, weight_series, cost_terms,
                         assess, assess_obstacles, assess_r2, assess_candidates)

    def _batch_arrays(self, frenet_states, target_speed, dynamic_obstacles=None, distribution=None,
                      static_obstacles=None, constraint_overrides=None, limits=None, max_stop_distance=None, route=None,
                      **run):
        """(the checked inputs of `plan_batch`, its remaining keywords)."""
        mode, dyn = _lib.FOT_DYN_NONE, None
        if distribution is not None and np.size(distribution) > 0:
            mode, dyn = _lib.FOT_DYN_DISTRIBUTION, np.asarray(distribution, dtype=np.float64)
        elif dynamic_obstacles is not None and np.size(dynamic_obstacles) > 0:
            mode, dyn = _lib.FOT_DYN_SINGLE, np.asarray(dynamic_obstacles, dtype=np.float64)[:, None]
        if limits is None:
            limits = self.resolve_limits(constraint_overrides)
        q = query_arrays(frenet_states, target_speed, limits, max_stop_distance, static_obstacles, dyn, mode, self.d_t_s)
        q.route = route_array(route, len(q.frenet), len(self.routes))
        return q, run

    def plan_batch_from_ego(self, ego, target_speed, last_kappa=0.0, converter: Optional[BatchCoordinateConverter] = None,
                            **kwargs):
        """plan() for n_q ego states at once: ego [n_q,5] (x, y, yaw, v, a), last_kappa scalar or [n_q] (the ego
        curvature plan() keeps between calls), `converter` the n_q nearest-point caches to use and update (row q for
        ego q; None: fresh ones on this planner's device, as a first plan() call has, each on the query's route when
        **kwargs has `route`).  The nearest-point search runs on the device (DESIGN.md section 4e), the rest of the
        Frenet conversion on the host, then `plan_batch` with **kwargs.  Returns (SweepResult, ok): where ok is False the conversion failed and plan() would return None --
        best_idx -1, best_cost inf, stats zero, winner_len 0 (`SweepResult.blank`)."""
        ego = np.asarray(ego, dtype=np.float64).reshape(-1, 5)
        n_q = ego.shape[0]
        q, run = self._batch_arrays(np.zeros((n_q, 6)), target_speed, **kwargs)    # checked before the device is used
        if converter is None and q.route is not None:
            converter = RoutedCoordinateConverter(self.routes, q.route, engine=self.engine)
        elif converter is None:
            converter = BatchCoordinateConverter(self.csp, n_q, engine=self.engine)
        else:
            # the converter's rows must search the paths the queries plan on: a row converted on one path and planned
            # on another would be a wrong Frenet state, not an error
            want = np.zeros(n_q, dtype=np.int64) if q.route is None else q.route.astype(np.int64)
            have = converter.route[:n_q] if isinstance(converter, RoutedCoordinateConverter) else np.zeros(n_q, np.int64)
            if not np.array_equal(have, want):
                raise ValueError("converter routes differ from the queries' route: pass a RoutedCoordinateConverter "
                                 "over this planner's routes with the same route array (rows on route 0 only: a "
                                 "BatchCoordinateConverter)")
        kappa = np.broadcast_to(np.asarray(last_kappa, dtype=np.float64), (n_q,))
        frenet, ok = ego_to_frenet_many(converter, np.arange(n_q), ego, kappa)
        q.frenet[:] = frenet
        res = self._run(q, **run)
        res.blank(~ok)
        return res, ok


class DeviceBatch:
    """A batch whose inputs and outputs live in torch CUDA tensors (buffers only): the timed
    region of `bench.py`'s device-resident leg calls `launch()` and nothing else.

    top_k > 0: every launch also writes the per-candidate table and ranks it (fot_rank_candidates) into
    out["rank_idx"] / out["rank_cost"] [n_q, top_k] and, with rank_series, out["rank_len"] [n_q, top_k] and
    out["rank_series"] [n_q, top_k, 15, n_t_max].

    cost_weights [n_w, 6] (every query) or [n_q, n_w, 6] (a list per query), columns _lib.COST_WEIGHT_KEYS: every
    launch also writes the per-candidate categories (shared with top_k) and selects each query's winner under every
    weighting (fot_select_weighted) into out["w_idx"] / out["w_cost"] [n_q, n_w] and, with weight_series,
    out["w_len"] [n_q, n_w] and out["w_series"] [n_q, n_w, 15, n_t_max].  cost_terms: out["cost_terms"]
    [n_q, stride, 5] = (Jp, Jd, Js, Jv, Jt) of every candidate (fot_cost_terms).

    assess: every launch also assesses its winners -- or, with top_k > 0 and rank_series, its ranked alternatives, of
    which rank 0 is the winner -- against an obstacle field (fot_assess_trajectories, DESIGN.md section 4i) into
    out["a_<name>"] for the names of engine.ASSESS_FIELDS, [n_q, m, ...] with m = 1 or top_k.  The field is the batch's
    own (dyn and static obstacles), or assess_obstacles [n_q, S, P, T, 2] (a NumPy array or a CUDA tensor, read as S
    samples of P pedestrians) with the batch's static obstacles.  assess_r2: threshold pairs (r2_dyn, r2_static), one
    or [n_r, 2]; None: the handle's own pair for that field (`SweepEngine.own_radii`), under which a trajectory is
    collision-free iff static_hit == 0 and dyn_hits <= floor(chance_epsilon * S).

    assess_candidates: every launch also assesses every generated candidate of every query -- regenerated on the
    device, never stored (fot_assess_candidates, DESIGN.md section 4j) -- against the same field and threshold pairs
    into out["ca_<name>"] [n_q, stride, ...] for the names of engine.ASSESS_FIELDS and out["ca_keep"] [n_q, stride],
    column i candidate i in generation order.  candidate_table: also write the per-candidate categories and costs
    (for `sweep_result(want_candidates=True)` without top_k)."""

    def __init__(self, planner: FrenetPlanner, frenet_states, target_speed, dyn, dyn_mode, limits=None,
                 max_stop_distance=None, static_obstacles=None, top_k: int = 0, rank_series: bool = True,
                 cost_weights=None, weight_series: bool = True, cost_terms: bool = False, route=None,
                 assess: bool = False, assess_obstacles=None, assess_r2=None, assess_candidates: bool = False,
                 candidate_table: bool = False):
        import torch
        q = query_arrays(frenet_states, target_speed, planner.resolve_limits(None) if limits is None else limits,
                         max_stop_distance, static_obstacles, dyn, dyn_mode, planner.d_t_s)
        n_q = len(q.frenet)
        route = route_array(route, n_q, len(planner.routes))
        self.top_k = int(top_k)
        if self.top_k > _lib.FOT_MAX_RANKED:
            raise ValueError(f"top_k must be in [1, {_lib.FOT_MAX_RANKED}]")
        weights, per_query = _weight_table(cost_weights, n_q)
        self.assess = bool(assess)
        self.assess_candidates = bool(assess_candidates)
        any_assess = self.assess or self.assess_candidates
        a_obs, a_mode = _assess_field(assess_obstacles, n_q) if any_assess else (None, None)
        a_mode = q.dyn_mode if a_obs is None else a_mode
        a_r2 = assess_radii(assess_r2) if any_assess and assess_r2 is not None else None
        self.n_w = 0 if weights is None else weights.shape[-2]
        eng = planner.engine
        dev = torch.device("cuda", eng.device)
        self.engine, self.n_q = eng, n_q
        self.n_v_host, self.frenet_host = q.n_v, q.frenet
        # the inputs on the device; a torch dyn stays where it is
        self.t = {key: a if isinstance(a, torch.Tensor) else torch.from_numpy(a).to(dev)
                  for key in ("frenet", "target", "limits", "stop", "v_grid", "n_v", "static", "dyn")
                  if (a := getattr(q, key)) is not None}
        if route is not None:
            self.t["route"] = torch.from_numpy(route).to(dev)
        self.batch = fot_batch(dataclasses.replace(q, **self.t), torch.Tensor.data_ptr)
        # the whole winner block in one contiguous buffer (what the sharded sweep gathers with one collective)
        self.block = WinnerBlock(n_q, eng.n_t_max, device=dev)
        self.out = dict(self.block.views)
        self.stride = eng.lib.fot_candidate_count(eng._h, int(self.batch.n_v_max), 1)

        def new(where: dict, key: str, shape, dtype) -> int:
            where[key] = torch.empty(shape, dtype=dtype, device=dev)
            return where[key].data_ptr()

        def selections(prefix: str, m: int, series: bool, s):      # s: a FotRanked or FotWeighted
            s.idx = new(self.out, prefix + "_idx", (n_q, m), torch.int32)
            s.cost = new(self.out, prefix + "_cost", (n_q, m), torch.float64)
            if series:
                s.len = new(self.out, prefix + "_len", (n_q, m), torch.int32)
                s.series = new(self.out, prefix + "_series", (n_q, m, _lib.FOT_N_SERIES, eng.n_t_max), torch.float64)
            return s

        if self.top_k > 0 or self.n_w > 0 or candidate_table:
            new(self.t, "cand_cat", (n_q, self.stride), torch.uint8)
        if self.top_k > 0 or candidate_table:
            new(self.t, "cand_cost", (n_q, self.stride), torch.float64)
            self.ranked = selections("rank", self.top_k, rank_series, _lib.FotRanked(k=self.top_k))
        if self.n_w > 0:
            self.t["weights"] = torch.from_numpy(weights).to(dev)
            self.weighted = selections("w", self.n_w, weight_series,
                                       _lib.FotWeighted(n_w=self.n_w, per_query=per_query,
                                                        weights=self.t["weights"].data_ptr()))
        self.cost_terms = bool(cost_terms)
        if self.cost_terms:
            new(self.out, "cost_terms", (n_q, self.stride, 5), torch.float64)
        if any_assess:
            self.assess_field = _lib.FotBatch.from_buffer_copy(self.batch)
            if a_obs is not None:
                self.t["a_dyn"] = a_obs.to(dev).contiguous() if isinstance(a_obs, torch.Tensor) else torch.from_numpy(a_obs).to(dev)
                f = self.assess_field
                f.dyn, f.dyn_mode = self.t["a_dyn"].data_ptr(), _lib.FOT_DYN_DISTRIBUTION
                f.S, f.P, f.T_obs = a_obs.shape[1], a_obs.shape[2], a_obs.shape[3]
            r2 = eng.own_radii(a_mode) if a_r2 is None else a_r2
            self.t["a_r2"] = torch.from_numpy(r2).to(dev)
        if self.assess:
            ranked = self.top_k > 0 and rank_series
            m, n_r = (self.top_k if ranked else 1), r2.shape[0]
            a = _lib.FotAssessed(m=m, n_t=eng.n_t_max, n_r=n_r, r2=self.t["a_r2"].data_ptr())
            a.series = self.out["rank_series" if ranked else "winner"].data_ptr()
            a.len = self.out["rank_len" if ranked else "winner_len"].data_ptr()
            for name, dt, shape in ASSESS_FIELDS:
                setattr(a, name, new(self.out, "a_" + name, (n_q, m, *(n_r if d == "r" else d for d in shape)),
                                     getattr(torch, dt)))
            self.assessed = a
        if self.assess_candidates:
            n_r = self.t["a_r2"].shape[0]
            a = _lib.FotAssessed(m=self.stride, n_t=0, n_r=n_r, r2=self.t["a_r2"].data_ptr())
            for name, dt, shape in ASSESS_FIELDS:
                setattr(a, name, new(self.out, "ca_" + name, (n_q, self.stride, *(n_r if d == "r" else d for d in shape)),
                                     getattr(torch, dt)))
            new(self.out, "ca_keep", (n_q, self.stride), torch.int32)
            self.cand_assessed = a
        self.result = fot_result(dict(self.out, **self.t), torch.Tensor.data_ptr)

    def launch(self, stream: Optional[int] = None) -> None:
        """Enqueue prepass + sweep + winner kernels on `stream` (raw cudaStream_t).  None: torch's current stream
        of the batch's device -- ordered behind whatever torch work produced the input tensors -- synchronised
        before returning."""
        if stream is None:
            import torch
            cur = torch.cuda.current_stream(self.out["best_idx"].device)
            self._enqueue(cur.cuda_stream or None)
            cur.synchronize()
            return
        self._enqueue(stream)

    def _route_ptr(self):
        r = self.t.get("route")
        return None if r is None else r.data_ptr()

    def _enqueue(self, stream) -> None:
        with self.engine.routes_bound(self._route_ptr()):
            self.engine.run_device(self.batch, self.result, stream)
            if self.top_k > 0:
                r = self.result
                self.engine.rank_device(self.batch, r.cand_cat, r.cand_cost, r.cand_stride, self.ranked, stream)
            if self.n_w > 0:
                self.engine.select_weighted_device(self.batch, self.result.cand_cat, self.stride, self.weighted, stream)
            if self.cost_terms:
                self.engine.cost_terms_device(self.batch, self.stride, self.out["cost_terms"].data_ptr(), stream)
            if self.assess:
                self.engine.assess_device(self.assess_field, self.assessed, stream)
            if self.assess_candidates:
                self.engine.assess_candidates_device(self.batch, self.assess_field, self.stride, self.cand_assessed,
                                                     self.out["ca_keep"].data_ptr(), stream)

    def sweep_result(self, want_candidates: bool = False, winner_samples: int = 0) -> SweepResult:
        """Host copy of the outputs of the last launch, once it has finished (launch() without a stream waits), as a
        SweepResult: the candidate table only with want_candidates, which needs top_k > 0 (or cost_weights, for the
        categories alone); winner_samples = k > 0: the first k samples of each winner series."""
        host = {k: v.cpu().numpy() for k, v in self.out.items()}
        assessed = {name: host.pop("a_" + name) for name, _, _ in ASSESS_FIELDS} if self.assess else None
        cand_assessed = {name: host.pop("ca_" + name) for name in (*(f[0] for f in ASSESS_FIELDS), "keep")} \
            if self.assess_candidates else None
        res = SweepResult(**host)
        res.assessed = assessed
        res.cand_assessed = cand_assessed
        if winner_samples and winner_samples > 0:
            res.winner = np.ascontiguousarray(res.winner[:, :, :min(int(winner_samples), res.winner.shape[2])])
        if want_candidates:
            res.cand_cat = self.t["cand_cat"].cpu().numpy()
            res.cand_cost = self.t["cand_cost"].cpu().numpy() if "cand_cost" in self.t else None
        return self.engine.finish_result(res, self.frenet_host, self.n_v_host)

    def launch_to_host(self, host_out: dict, stream: Optional[int] = None, winner_samples: int = 0) -> None:
        """fot_plan_batch_device_to_host: sweep the (device-resident) batch and deliver the winners into the host
        arrays of `host_out` (keys of `self.out`; torch CPU tensors or NumPy arrays, ideally page-locked): the
        queries run in ranges and each range's winners are copied back while the next range is swept.  `stream`:
        the raw cudaStream_t on which the batch's inputs become ready (None: they are ready).  `winner_samples = k > 0`:
        only the first k samples of every winner series come back (`host_out["winner"]` is [n_q, 15, k]) -- what a
        closed-loop caller consumes (integrated_simulator.py:663), 240 B instead of 6.1 KB per query at k = 2.
        Ranked, weighted and assessed outputs do not come back through this call: a batch with top_k > 0,
        cost_weights, cost_terms, assess or assess_candidates raises ValueError."""
        if self.top_k > 0:
            raise ValueError("launch_to_host does not return ranked outputs; use launch() with top_k > 0")
        if self.assess:
            raise ValueError("launch_to_host does not return assessments; use launch() with assess=True")
        if self.assess_candidates:
            raise ValueError("launch_to_host does not return candidate assessments; use launch() with assess_candidates=True")
        if self.n_w > 0 or self.cost_terms:
            raise ValueError("launch_to_host does not return weighted outputs or cost terms; use launch()")
        import ctypes as C
        ptr = lambda a: a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data
        r = fot_result(host_out, ptr, winner_samples)
        with self.engine.routes_bound(self._route_ptr()):
            _lib.check(self.engine.lib.fot_plan_batch_device_to_host(self.engine._h, C.byref(self.batch), C.byref(r),
                                                                     C.c_void_p(stream) if stream else None),
                       "fot_plan_batch_device_to_host")

    def dense_evals(self) -> int:
        """Densely credited point-vs-obstacle tests of this batch (SURVEY.md section 8d)."""
        pts = self.engine.points_per_query(self.frenet_host, self.n_v_host)
        n_circ = max(1, self.engine.n_circles)
        per_point = self.batch.S * self.batch.P + self.batch.n_static
        return int(pts.sum()) * n_circ * int(per_point)


def _assess_field(obstacles, n_q: int):
    """(assess_obstacles as a float64 [n_q, S, P, T, 2] NumPy array or torch tensor, or None; the dyn mode the handle's
    own threshold pair is taken for).  Raises ValueError on any other shape or dtype."""
    if obstacles is None:
        return None, None
    if hasattr(obstacles, "data_ptr"):
        import torch
        a, f64 = obstacles, torch.float64
    else:
        a, f64 = np.ascontiguousarray(obstacles, dtype=np.float64), np.float64
    if a.ndim != 5 or a.shape[0] != n_q or a.shape[-1] != 2 or a.dtype != f64 or min(a.shape) < 1:
        raise ValueError(f"assess_obstacles must be float64 [n_q={n_q}, S, P, T, 2] with S, P, T >= 1, "
                         f"got {a.dtype} {list(a.shape)}")
    return a, _lib.FOT_DYN_DISTRIBUTION


def _weight_table(cost_weights, n_q: int):
    """cost_weights as a contiguous float64 array and its fot_weighted_t.per_query flag: [n_w, 6] -> 0 (one list for
    every query), [n_q, n_w, 6] -> 1; None -> (None, 0).  Raises ValueError on any other shape or n_w outside
    [1, FOT_MAX_WEIGHT_SETS]."""
    if cost_weights is None:
        return None, 0
    w = np.ascontiguousarray(cost_weights, dtype=np.float64)
    n_k = len(_lib.COST_WEIGHT_KEYS)
    if w.ndim == 2 and w.shape[1] == n_k:
        per_query = 0
    elif w.ndim == 3 and w.shape[0] == n_q and w.shape[2] == n_k:
        per_query = 1
    else:
        raise ValueError(f"cost_weights must be [n_w, {n_k}] or [n_q={n_q}, n_w, {n_k}], got {list(w.shape)}")
    if not 1 <= w.shape[-2] <= _lib.FOT_MAX_WEIGHT_SETS:
        raise ValueError(f"the number of weightings must be in [1, {_lib.FOT_MAX_WEIGHT_SETS}], got {w.shape[-2]}")
    return w, per_query


class WinnerBlock:
    """A rank's winner block for `cap` queries in ONE contiguous buffer: best_idx | winner_len | stats | best_cost |
    winner, each section 256-byte aligned (what `gather_winners` moves with one collective, SURVEY.md section 8e:
    about 6.2 KB per query).  `views[key]` are typed tensors into the buffer; the kernels write straight into them."""

    def __init__(self, cap: int, n_t_max: int, device=None, sections=None):
        import torch
        self.cap = int(cap)
        self.sections = sections or winner_fields(n_t_max)
        self.offsets, off = {}, 0
        for key, dt, shape in self.sections:
            n = self.cap * int(np.prod(shape, dtype=np.int64)) * torch.empty((), dtype=dt).element_size()
            self.offsets[key] = (off, n)
            off = (off + n + 255) // 256 * 256
        self.nbytes = max(off, 256)
        self.buf = torch.empty(self.nbytes, dtype=torch.uint8, device=device)
        self.views = self.unpack(self.buf)

    def unpack(self, buf):
        """Typed views of a buffer laid out like this block (leading dims of `buf` are kept: [world, nbytes] ->
        [world, cap, ...])."""
        lead = tuple(buf.shape[:-1])
        out = {}
        for key, dt, shape in self.sections:
            off, n = self.offsets[key]
            out[key] = buf[..., off:off + n].contiguous().view(dt).reshape(lead + (self.cap,) + tuple(shape)) if lead \
                else buf[off:off + n].view(dt).reshape((self.cap,) + tuple(shape))
        return out


def gather_winners(out: dict, group=None, counts=None) -> dict:
    """The one collective of the sharded sweep: every rank's winner block (best_idx, best_cost, stats, winner_len,
    winner -- any dict of tensors with the queries on dim 0) packed into ONE contiguous buffer and moved by ONE
    `all_gather_into_tensor` over the process group (NCCL on GPUs, gloo in the CPU tests); returns the blocks of all
    ranks concatenated in rank order.

    Ranks may hold different numbers of queries (`shard_bounds` gives the last rank a shorter or empty block): every
    block is padded to the longest one and the padding is trimmed after the gather.  `counts` = queries per rank when
    the caller knows them (e.g. from `shard_bounds`); otherwise they are exchanged first (one extra, 8-byte
    collective).  A `WinnerBlock`'s views are gathered without the packing copy when its capacity already equals the
    longest block."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return out
    world = dist.get_world_size(group)
    first = next(iter(out.values()))
    n_local, dev = int(first.shape[0]), first.device
    if counts is None:
        mine = torch.tensor([n_local], dtype=torch.int64, device=dev)
        allc = torch.empty(world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allc, mine, group=group)
        counts = [int(c) for c in allc.cpu()]
    counts = [int(c) for c in counts]
    assert len(counts) == world and counts[dist.get_rank(group)] == n_local, (counts, n_local)
    per = max(counts)
    sections = tuple((k, t.dtype, tuple(t.shape[1:])) for k, t in out.items())
    blk = WinnerBlock(per, 0, device=dev, sections=sections)
    own = getattr(first, "_base", None)
    zero_copy = per == n_local and own is not None and own.dtype == torch.uint8 and own.numel() == blk.nbytes and \
        all(t._base is own and t.data_ptr() == own.data_ptr() + blk.offsets[k][0] for k, t in out.items())
    if zero_copy:
        send = own
    else:
        send = blk.buf
        send.zero_()
        for k, t in out.items():
            blk.views[k][:n_local].copy_(t)
    gathered = torch.empty((world, blk.nbytes), dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(gathered.view(-1), send, group=group)
    parts = blk.unpack(gathered)
    if all(c == per for c in counts):
        return {k: v.reshape((world * per,) + tuple(v.shape[2:])) for k, v in parts.items()}
    return {k: torch.cat([v[r, :counts[r]] for r in range(world)], dim=0) for k, v in parts.items()}


class _RawCuda:
    """A raw device pointer as something torch can wrap (`torch.as_tensor(obj, device=...)`)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


class PeerGather:
    """The one gather of the query-sharded sweep without a collective call: every rank's winner block lands in the
    ROOT's memory, stored there by that rank's own `fot_winner` kernel through NVLink peer memory
    (fot_set_result_mirror), while the rank's next sweep is already running.

    The root owns `depth` buffers of `world x WinnerBlock(cap)` bytes (fot_peer_alloc) and a flag word per rank; the
    other ranks map them (CUDA IPC handle -> fot_peer_open; the 64-byte handles travel through torch.distributed).
    Step k of every rank is mirrored into buffer k % depth, slice `rank`; behind it the rank publishes k + 1 in its flag
    word.  `await_step(k)` on the root enqueues a device-side wait for all flags; `views(k)` are typed tensors
    [world, cap, ...] into the buffer.  One process per GPU, one handle per process.
    """

    def __init__(self, engine: SweepEngine, cap: int, group=None, root: int = 0, depth: int = 2):
        import ctypes as C
        import torch
        import torch.distributed as dist
        self.engine, self.lib, self.root, self.depth = engine, engine.lib, int(root), int(depth)
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.dev = torch.device("cuda", engine.device)
        self.layout = WinnerBlock(cap, engine.n_t_max, device="meta")             # offsets only
        self.nbytes = self.layout.nbytes
        self.flag_bytes = 256 * ((4 * self.world + 255) // 256)
        total = self.depth * self.world * self.nbytes + self.flag_bytes + 256
        handle = torch.zeros(64, dtype=torch.uint8)
        self._base = C.c_void_p()
        self._owned = self.rank == self.root
        if self._owned:
            buf = C.create_string_buffer(64)
            _lib.check(self.lib.fot_peer_alloc(engine.device, total, C.byref(self._base), buf), "fot_peer_alloc")
            handle = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).clone()
        h_dev = handle.to(self.dev)
        dist.broadcast(h_dev, src=dist.get_global_rank(group, self.root) if group is not None else self.root, group=group)
        if not self._owned:
            raw = bytes(h_dev.cpu().numpy().tobytes())
            _lib.check(self.lib.fot_peer_open(engine.device, raw, C.byref(self._base)), "fot_peer_open")
        self.base = int(self._base.value)
        self.flags_ptr = self.base + self.depth * self.world * self.nbytes
        self.err_ptr = self.flags_ptr + self.flag_bytes
        self.step = 0

    def _slice_ptr(self, k: int, rank: int) -> int:
        return self.base + ((k % self.depth) * self.world + rank) * self.nbytes

    def attach(self, k: Optional[int] = None) -> None:
        """The engine's next fot_plan_batch_device launch mirrors its winner block into buffer k % depth (default: the
        running step counter, which then advances)."""
        import ctypes as C
        if k is None:
            k = self.step
            self.step += 1
        p = self._slice_ptr(k, self.rank)
        m = fot_result({key: p + off for key, (off, _) in self.layout.offsets.items()}, int)
        _lib.check(self.lib.fot_set_result_mirror(self.engine._h, C.byref(m), C.c_void_p(self.flags_ptr + 4 * self.rank)),
                   "fot_set_result_mirror")

    def detach(self) -> None:
        _lib.check(self.lib.fot_set_result_mirror(self.engine._h, None, None), "fot_set_result_mirror")

    def await_step(self, seq: int, stream: Optional[int] = None) -> None:
        """Root: enqueue a wait until every rank has published launch number `seq` (1-based count of its mirrored
        launches)."""
        import ctypes as C
        assert self._owned, "await_step is a root-side call"
        _lib.check(self.lib.fot_peer_await(self.engine.device, C.c_void_p(stream) if stream else None, C.c_void_p(self.flags_ptr),
                                           self.world, int(seq), C.c_void_p(self.err_ptr)), "fot_peer_await")

    def views(self, k: int) -> dict:
        """Root: the gathered blocks of step k as tensors [world, cap, ...] (views into the peer buffer)."""
        import torch
        assert self._owned
        raw = torch.as_tensor(_RawCuda(self._slice_ptr(k, 0), self.world * self.nbytes), device=self.dev)
        return self.layout.unpack(raw.view(self.world, self.nbytes))

    def timed_out(self) -> bool:
        import torch
        assert self._owned
        return bool(torch.as_tensor(_RawCuda(self.err_ptr, 4), device=self.dev).view(torch.int32).item())

    def close(self) -> None:
        if self._base is not None and self._base.value:
            self.detach()
            if self._owned:
                self.lib.fot_peer_free(self._base)
            else:
                self.lib.fot_peer_close(self._base)
            self._base = None
