"""Evaluation image metrics on the device: MSE, PSNR, SSIM and MS-SSIM in one fused pass per scale (rdg_image_metrics).

These are the metrics the reference reports for held-out views (RoDyGSEvaluator.eval, VizScoreEvaluator, through piqa):
an 11x11 Gaussian window (sigma 1.5) over the VALID region only, averaged per channel, and MS-SSIM over five scales.  They
are not the training SSIM in SplatTrainStep.loss_parts[2], which zero-pads the window over the full image and gives a
lower number near the borders.  piqa's conventions are recalled, not pinned against piqa itself: INTEGRATION.md,
"Scoring held-out views", states them.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import check, ptr


def image_metrics(pred: torch.Tensor, gt: torch.Tensor, value_range: float = 1.0) -> torch.Tensor:
    """(mse, psnr, ssim, ms_ssim) of every image pair as a [B, 4] float32 tensor on the inputs' device, without a host read.

    pred, gt: [C, H, W] or [B, C, H, W] CUDA tensors of the same shape, H, W >= 11; other dtypes are converted to float32.
    psnr = 10 log10(value_range^2 / (mse + 1e-8)); SSIM's constants are (0.01 value_range)^2 and (0.03 value_range)^2.
    ms_ssim is NaN for images smaller than 161 pixels on a side (its fifth scale must still hold the window); the other
    three columns are computed for every size.  Not differentiable.  The result of an image does not depend on the
    other images of the batch, and repeated calls give identical bits."""
    for name, t in (("pred", pred), ("gt", gt)):
        if not torch.is_tensor(t):
            raise TypeError(f"image_metrics: {name} must be a tensor, got {type(t).__name__}")
        if not t.is_cuda:
            raise RuntimeError(f"image_metrics: {name} is on {t.device}; rodygs_b200 runs on CUDA tensors only (no CPU fallback)")
        if t.dim() not in (3, 4):
            raise ValueError(f"image_metrics: {name} must be [C, H, W] or [B, C, H, W], got shape {tuple(t.shape)}")
    if pred.shape != gt.shape:
        raise ValueError(f"image_metrics: pred has shape {tuple(pred.shape)} but gt has {tuple(gt.shape)}")
    if pred.device != gt.device:
        raise ValueError(f"image_metrics: pred is on {pred.device} but gt on {gt.device}")
    H, W = pred.shape[-2:]
    if H < 11 or W < 11:
        raise ValueError(f"image_metrics: pred and gt are {H}x{W}; the 11x11 SSIM window needs H and W >= 11")
    value_range = float(value_range)
    if not value_range > 0.0:
        raise ValueError(f"image_metrics: value_range must be > 0, got {value_range}")
    x, y = (t.detach() if t.dim() == 4 else t.detach()[None] for t in (pred, gt))
    x, y = (t.to(torch.float32).contiguous() for t in (x, y))
    B, C = x.shape[:2]
    lib = _lib.load()
    nbytes = int(lib.rdg_image_metrics_workspace_bytes(B, C, H, W))
    if nbytes < 0:
        check(nbytes)
    with torch.cuda.device(x.device):
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        out = torch.empty(B, 4, dtype=torch.float32, device=x.device)
        check(lib.rdg_image_metrics(ptr(x), ptr(y), B, C, H, W, value_range, ptr(out), ptr(ws), nbytes, _lib.stream_ptr()))
    return out
