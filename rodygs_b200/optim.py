"""Adam on the flat parameter buffer with the reference's parameter groups (SURVEY.md §8 f1).

Mirror of ThreeDGSTrainer.optim_setup / update_learning_rate
(/root/reference/src/trainer/rodygs_static.py:106-149), DynTrainer.append_motion_optim
(/root/reference/src/trainer/rodygs_dynamic.py:92-123) and get_expon_lr_func
(/root/reference/src/utils/general_utils.py:40-73).  One CUDA launch per optimiser step
(rdg_adam_groups); the deformation MLP (68 K parameters) stays with torch.optim.Adam.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import torch

from . import _lib
from ._lib import check, ptr

# flat-layout field -> the reference's group name
GROUP_OF = {"xyz": "xyz", "features_dc": "f_dc", "features_rest": "f_rest", "opacity": "opacity", "scaling": "scaling",
            "rotation": "rotation"}


def expon_lr(step: int, lr_init: float, lr_final: float, lr_delay_steps: int = 0, lr_delay_mult: float = 1.0,
             max_steps: int = 1000000) -> float:
    """get_expon_lr_func(...)(step) (general_utils.py:40-73): log-linear decay with an optional eased-in start."""
    if step < 0 or (lr_init == 0.0 and lr_final == 0.0):
        return 0.0
    if lr_delay_steps > 0:
        delay_rate = lr_delay_mult + (1 - lr_delay_mult) * math.sin(0.5 * math.pi * min(max(step / lr_delay_steps, 0.0), 1.0))
    else:
        delay_rate = 1.0
    t = min(max(step / max_steps, 0.0), 1.0)
    return delay_rate * math.exp(math.log(lr_init) * (1 - t) + math.log(lr_final) * t)


@dataclass
class GaussianLRs:
    """train_kubric_mrig.yaml:159-167 (static) / :236-260 (dynamic: scaling_lr 0.001, motion_coeff_lr 1.6e-4)."""
    position_lr_init: float = 0.00016
    position_lr_final: float = 1.6e-06
    position_lr_delay_mult: float = 0.01
    position_lr_max_steps: int = 20000
    feature_lr: float = 0.0025
    opacity_lr: float = 0.05
    scaling_lr: float = 0.005
    rotation_lr: float = 0.001
    motion_coeff_lr: Optional[float] = None      # dynamic model only

    def group_lrs(self, iteration: int, spatial_lr_scale: float) -> Dict[str, float]:
        """Learning rate of every group at `iteration` (only xyz is scheduled, rodygs_static.py:143-149)."""
        lrs = {
            "xyz": expon_lr(iteration, self.position_lr_init * spatial_lr_scale, self.position_lr_final * spatial_lr_scale,
                            lr_delay_mult=self.position_lr_delay_mult, max_steps=self.position_lr_max_steps),
            "f_dc": self.feature_lr, "f_rest": self.feature_lr / 20.0, "opacity": self.opacity_lr,
            "scaling": self.scaling_lr, "rotation": self.rotation_lr,
        }
        if self.motion_coeff_lr is not None:
            lrs["motion_coeff"] = self.motion_coeff_lr
        return lrs


@dataclass
class CameraLRs:
    """Learning rates of the training-camera table (SplatTrainStep.enable_camera_learning): lr_q for the quaternions, lr_T for
    the translations, both scaled by the warmup + cosine factor

        f(it) = min(1, it / warmup_steps) * (final_ratio + (1 - final_ratio) * 0.5 * (1 + cos(pi * p))),
        p = clamp((it - warmup_steps) / (max_steps - warmup_steps), 0, 1)

    (f = 1 for the warmup factor when warmup_steps = 0).  The formula of the reference's CameraQuatOptimizer is recalled, not
    pinned (INTEGRATION.md "Learning the training cameras"), and its default values are not known: the two rates are
    required, and the other defaults give constant rates."""
    lr_q: float
    lr_T: float
    warmup_steps: int = 0
    max_steps: int = 1
    final_ratio: float = 1.0

    def __post_init__(self):
        for name in ("lr_q", "lr_T", "final_ratio"):
            v = float(getattr(self, name))
            if not (v >= 0.0 and math.isfinite(v)):
                raise ValueError(f"CameraLRs: {name} must be a finite value >= 0, got {getattr(self, name)}")
        if int(self.warmup_steps) != self.warmup_steps or self.warmup_steps < 0:
            raise ValueError(f"CameraLRs: warmup_steps must be an integer >= 0, got {self.warmup_steps}")
        if int(self.max_steps) != self.max_steps or self.max_steps <= self.warmup_steps:
            raise ValueError(f"CameraLRs: max_steps must be an integer > warmup_steps, got {self.max_steps}")

    def factor(self, it: int) -> float:
        warm = 1.0 if self.warmup_steps == 0 else min(1.0, it / self.warmup_steps)
        p = min(max((it - self.warmup_steps) / (self.max_steps - self.warmup_steps), 0.0), 1.0)
        return warm * (self.final_ratio + (1.0 - self.final_ratio) * 0.5 * (1.0 + math.cos(math.pi * p)))

    def rates(self, it: int) -> Tuple[float, float]:
        """(lr_q, lr_T) at iteration `it`."""
        f = self.factor(it)
        return self.lr_q * f, self.lr_T * f


class GaussianAdam:
    """torch.optim.Adam(groups, lr=0.0, eps=1e-15) of ONE model ("static" or "dynamic") living in the flat buffers
    of a SplatTrainStep.  `ranges`: reference group name -> (float offset, numel) inside those buffers."""

    def __init__(self, ranges: Dict[str, Tuple[int, int]], total: int, lrs: GaussianLRs, spatial_lr_scale: float,
                 device="cuda", betas=(0.9, 0.999), eps: float = 1e-15):
        self.ranges = dict(ranges)
        self.lrs, self.spatial_lr_scale = lrs, float(spatial_lr_scale)
        self.betas, self.eps = betas, eps
        self.exp_avg = torch.zeros(total, dtype=torch.float32, device=device)
        self.exp_avg_sq = torch.zeros(total, dtype=torch.float32, device=device)
        self.steps = 0

    def moments(self, name: str) -> Tuple[torch.Tensor, torch.Tensor]:
        off, n = self.ranges[name]
        return self.exp_avg[off:off + n], self.exp_avg_sq[off:off + n]

    def step(self, params: torch.Tensor, grads: torch.Tensor, iteration: int, grad_scale: float = 1.0, skip=()):
        """update_learning_rate(iteration) + optimizer.step() (rodygs.py:209,364).  skip: group names another kernel has
        already stepped for this iteration (the SH groups, SplatTrainStep._sh_adam_from_factors)."""
        _lib.require_cuda(params, grads)
        if params.numel() != self.exp_avg.numel() or grads.numel() != params.numel():
            raise RuntimeError("optimizer state does not match the flat buffers (rebuild it after densification)")
        lr = self.lrs.group_lrs(iteration, self.spatial_lr_scale)
        live = [(name, off, n) for name, (off, n) in self.ranges.items() if n > 0 and name not in skip]
        arr = (_lib.RdgAdamGroup * len(live))()
        for k, (name, off, n) in enumerate(live):
            arr[k].begin, arr[k].end, arr[k].lr = off, off + n, lr[name]
        self.steps += 1
        if live:
            check(_lib.load().rdg_adam_groups(ptr(params), ptr(grads), ptr(self.exp_avg), ptr(self.exp_avg_sq), arr, len(live),
                                              self.betas[0], self.betas[1], self.eps, self.steps, float(grad_scale),
                                              _lib.stream_ptr()))
        return lr
