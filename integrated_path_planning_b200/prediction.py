"""The predictor's post-processing on the device (SURVEY.md section 8f, rank 1).

Mirrors the tail of the reference's prediction path -- `TrajectoryPredictor.predict_cv`,
`.process_prediction`, the closest-to-mean selection of `.predict_single_best`
(src/prediction/trajectory_predictor.py:188-353) and the t = 0 prepend of
`IntegratedSimulator._update_prediction` (src/simulation/integrated_simulator.py:503-525) -- for batches
of independent queries, with every tensor resident on the GPU.  The outputs are laid out exactly as
`fot_batch_t.dyn` wants them ([n_q][S][P][T_obs][2]), so a batched roll-out goes from "last two
observations" to "best trajectory per query" without the obstacle tensor ever crossing PCIe.

torch tensors are buffers only; the arithmetic is in libfot.so (csrc/fot_predict.cuh), bit-identical to
the reference's NumPy.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import numpy as np

from . import _lib


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class DevicePredictionPostprocessor:
    """Same knobs as TrajectoryPredictor.__init__ (trajectory_predictor.py:27-46)."""

    def __init__(self, pred_len: int = 12, sgan_dt: float = 0.4, sim_dt: float = 0.1, plan_horizon: float = 5.0,
                 device: int = 0):
        import torch
        self.lib = _lib.load()
        self.pred_len, self.sgan_dt, self.sim_dt, self.plan_horizon = int(pred_len), float(sgan_dt), float(sim_dt), float(plan_horizon)
        self.device = int(device)
        self._dev = torch.device("cuda", self.device)
        # the reference's own expression for the output grid (:214-215, :283-284), evaluated by NumPy
        target_horizon = max(self.plan_horizon, self.pred_len * self.sgan_dt)
        self.time_target_host = np.arange(self.sim_dt, target_horizon + 1e-9, self.sim_dt)
        self.n_steps = len(self.time_target_host)
        self.time_target = torch.from_numpy(self.time_target_host).to(self._dev)

    # -- helpers -------------------------------------------------------------------------------
    def _dev_f64(self, a, shape):
        import torch
        if a is None:
            return None
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))
        t = t.to(self._dev, dtype=torch.float64).contiguous()
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f"expected shape {tuple(shape)}, got {tuple(t.shape)}")
        return t

    def _stale(self, staleness, n_q):
        import torch
        if staleness is None:
            return None
        s = torch.as_tensor(staleness, dtype=torch.float64).reshape(-1)
        if s.numel() == 1:
            s = s.expand(n_q)
        return s.to(self._dev).contiguous()

    def _stream(self):
        """torch's current stream ON THIS OBJECT'S DEVICE (not on torch's current device)."""
        import torch
        return C.c_void_p(torch.cuda.current_stream(self._dev).cuda_stream)

    # -- API -----------------------------------------------------------------------------------
    def predict_cv(self, p_curr, p_prev=None, staleness=None, current_positions=None, out=None,
                   obs_float32: bool = False):
        """Constant-velocity obstacle tensor.  p_curr / p_prev [n_q, P, 2] (the last two observation
        samples, sgan_dt apart; p_prev None = zero velocity), staleness scalar or [n_q],
        current_positions [n_q, P, 2] or None.  Returns [n_q, 1, P, T, 2] on the device, T = n_steps
        (+ 1 with the t = 0 column); `out` re-uses a caller-owned buffer of that shape.  obs_float32: treat
        the observations as the float32 tensors the reference's observer hands its predictor (the simulator's
        real data flow); the default takes them as the float64 values given."""
        import torch
        n_q, P = p_curr.shape[0], p_curr.shape[1]
        pc = self._dev_f64(p_curr, (n_q, P, 2))
        pp = self._dev_f64(p_prev, (n_q, P, 2))
        cur = self._dev_f64(current_positions, (n_q, P, 2))
        st = self._stale(staleness, n_q)
        T = self.n_steps + (cur is not None)
        if out is None:
            out = torch.empty((n_q, 1, P, T, 2), dtype=torch.float64, device=self._dev)
        elif tuple(out.shape) != (n_q, 1, P, T, 2) or out.dtype != torch.float64 or not out.is_contiguous():
            raise ValueError("out must be a contiguous float64 tensor of shape [n_q, 1, P, T, 2]")
        _lib.check(self.lib.fot_predict_cv_device(self.device, self._stream(), n_q, P, _p(pc), _p(pp), _p(st), self.sgan_dt,
                                                  _p(self.time_target), self.n_steps, _p(cur), int(bool(obs_float32)), _p(out)),
                   "fot_predict_cv_device")
        return out

    def process_prediction(self, pred, anchor=None, staleness=None):
        """Resample raw predictions onto the planner grid.  pred [n_q, S, pred_len, P, 2], anchor
        [n_q, P, 2] or None.  Returns [n_q, S, P, n_steps, 2]."""
        import torch
        n_q, S, L, P = pred.shape[0], pred.shape[1], pred.shape[2], pred.shape[3]
        pr = self._dev_f64(pred, (n_q, S, L, P, 2))
        an = self._dev_f64(anchor, (n_q, P, 2))
        st = self._stale(staleness, n_q)
        out = torch.empty((n_q, S, P, self.n_steps, 2), dtype=torch.float64, device=self._dev)
        _lib.check(self.lib.fot_process_prediction_device(self.device, self._stream(), n_q, S, P, L, _p(pr), _p(an), _p(st),
                                                          self.sgan_dt, _p(self.time_target), self.n_steps, _p(out)),
                   "fot_process_prediction_device")
        return out

    def select_best(self, samples):
        """Index of the sample closest to the mean, per query.  samples [n_q, S, P, T, 2] -> int32 [n_q]."""
        import torch
        n_q, S, P, T = samples.shape[:4]
        sm = self._dev_f64(samples, (n_q, S, P, T, 2))
        dist = torch.empty((n_q, S), dtype=torch.float64, device=self._dev)
        best = torch.empty((n_q,), dtype=torch.int32, device=self._dev)
        _lib.check(self.lib.fot_select_best_sample_device(self.device, self._stream(), n_q, S, P, T, _p(sm), _p(dist), _p(best)),
                   "fot_select_best_sample_device")
        return best, dist

    def prepend_current(self, tensor, current_positions, pick=None, conditional=True):
        """t = 0 column.  tensor [n_q, S, P, T, 2]; pick int32 [n_q] selects one sample per query.
        Returns [n_q, 1 or S, P, T + 1, 2]."""
        import torch
        n_q, S, P, T = tensor.shape[:4]
        tn = self._dev_f64(tensor, (n_q, S, P, T, 2))
        cur = self._dev_f64(current_positions, (n_q, P, 2))
        out = torch.empty((n_q, 1 if pick is not None else S, P, T + 1, 2), dtype=torch.float64, device=self._dev)
        _lib.check(self.lib.fot_prepend_current_device(self.device, self._stream(), n_q, S, P, T, _p(tn), _p(pick), _p(cur),
                                                       int(bool(conditional)), _p(out)), "fot_prepend_current_device")
        return out

    def obstacles_from_samples(self, pred, anchor, staleness, current_positions) -> Tuple["object", "object", "object"]:
        """predict_single_best + _update_prediction for S raw samples per query: returns
        (representative sample [n_q, 1, P, T+1, 2], distribution [n_q, S, P, T+1, 2], best index [n_q])."""
        dense = self.process_prediction(pred, anchor, staleness)
        best, _ = self.select_best(dense)
        single = self.prepend_current(dense, current_positions, pick=best, conditional=True)
        dist = self.prepend_current(dense, current_positions, pick=None, conditional=False)
        return single, dist, best


def safety_metrics(ego, ped_pos, ped_vel, ego_radius: float, ped_radius: float, footprint=None, n_peds=None,
                   device: int = 0):
    """compute_safety_metrics_static (src/core/data_structures.py:301-388) for a batch of queries on the
    device.  ego [n_q, 5] (x, y, yaw, v, a), ped_pos / ped_vel [n_q, P, 2] (host arrays or CUDA tensors),
    n_peds optional [n_q], each in [0, P] (ValueError otherwise).  Returns a dict of CUDA tensors [n_q]:
    min_distance, collision (bool), ttc, clearance, clearance_ahead -- the inputs of
    FailSafeStateMachine.update / _get_planner_config."""
    import torch
    lib = _lib.load()
    dev = torch.device("cuda", int(device))
    f64 = lambda a: (a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))
                     ).to(dev, dtype=torch.float64).contiguous()
    ego_t, pos_t, vel_t = f64(ego).reshape(-1, 5), f64(ped_pos), f64(ped_vel)
    n_q, P = ego_t.shape[0], pos_t.shape[1]
    if tuple(pos_t.shape) != (n_q, P, 2) or tuple(vel_t.shape) != (n_q, P, 2):
        raise ValueError("ped_pos / ped_vel must be [n_q, P, 2]")
    np_t = None
    if n_peds is not None:
        # a count above P would read the next query's pedestrians (past the buffer for the last query)
        n = n_peds if isinstance(n_peds, torch.Tensor) else torch.as_tensor(np.asarray(n_peds))
        if tuple(n.shape) != (n_q,):
            raise ValueError(f"n_peds must be [n_q] = [{n_q}], got {tuple(n.shape)}")
        if bool(((n < 0) | (n > P)).any()):
            raise ValueError(f"n_peds must lie in [0, P] = [0, {P}]")
        np_t = n.to(dev, dtype=torch.int32).contiguous()
    if footprint is None:
        combined, offs, n_circ = float(ego_radius) + float(ped_radius), None, 0
    else:
        o = np.ascontiguousarray(footprint.offsets, dtype=np.float64).reshape(-1)
        combined, offs, n_circ = float(footprint.radius) + float(ped_radius), o.ctypes.data_as(_lib.c_double_p), o.size
    out = torch.empty((n_q, 5), dtype=torch.float64, device=dev)
    _lib.check(lib.fot_safety_metrics_device(int(device), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream), n_q, P,
                                             _p(ego_t), _p(pos_t) if P else None, _p(vel_t) if P else None, _p(np_t),
                                             combined, offs, n_circ, _p(out)), "fot_safety_metrics_device")
    return {"min_distance": out[:, 0], "collision": out[:, 1] > 0.5, "ttc": out[:, 2], "clearance": out[:, 3],
            "clearance_ahead": out[:, 4]}
