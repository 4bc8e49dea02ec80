"""Evaluation image metrics on the device: MSE, PSNR, SSIM and MS-SSIM in one fused pass per scale (rdg_image_metrics), and
their masked forms over a covisibility mask, mPSNR and mSSIM (rdg_masked_image_metrics).

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


def _pair(fn: str, pred: torch.Tensor, gt: torch.Tensor, value_range: float):
    """Checks shared by the metrics entry points: (x, y) as contiguous float32 [B, C, H, W], and value_range as a float."""
    for name, t in (("pred", pred), ("gt", gt)):
        if not torch.is_tensor(t):
            raise TypeError(f"{fn}: {name} must be a tensor, got {type(t).__name__}")
        if not t.is_cuda:
            raise RuntimeError(f"{fn}: {name} is on {t.device}; rodygs_b200 runs on CUDA tensors only (no CPU fallback)")
        if t.dim() not in (3, 4):
            raise ValueError(f"{fn}: {name} must be [C, H, W] or [B, C, H, W], got shape {tuple(t.shape)}")
    if pred.shape != gt.shape:
        raise ValueError(f"{fn}: pred has shape {tuple(pred.shape)} but gt has {tuple(gt.shape)}")
    if pred.device != gt.device:
        raise ValueError(f"{fn}: pred is on {pred.device} but gt on {gt.device}")
    H, W = pred.shape[-2:]
    if H < 11 or W < 11:
        raise ValueError(f"{fn}: pred and gt are {H}x{W}; the 11x11 SSIM window needs H and W >= 11")
    value_range = float(value_range)
    if not value_range > 0.0:
        raise ValueError(f"{fn}: value_range must be > 0, got {value_range}")
    x, y = (t.detach() if t.dim() == 4 else t.detach()[None] for t in (pred, gt))
    x, y = (t.to(torch.float32).contiguous() for t in (x, y))
    return x, y, value_range


def image_metrics(pred: torch.Tensor, gt: torch.Tensor, value_range: float = 1.0) -> torch.Tensor:
    """(mse, psnr, ssim, ms_ssim) of every image pair as a [B, 4] float32 tensor on the inputs' device, without a host read.

    pred, gt: [C, H, W] or [B, C, H, W] CUDA tensors of the same shape, H, W >= 11; other dtypes are converted to float32.
    psnr = 10 log10(value_range^2 / (mse + 1e-8)); SSIM's constants are (0.01 value_range)^2 and (0.03 value_range)^2.
    ms_ssim is NaN for images smaller than 161 pixels on a side (its fifth scale must still hold the window); the other
    three columns are computed for every size.  Not differentiable.  The result of an image does not depend on the
    other images of the batch, and repeated calls give identical bits."""
    x, y, value_range = _pair("image_metrics", pred, gt, value_range)
    B, C, H, W = x.shape
    lib = _lib.load()
    nbytes = int(lib.rdg_image_metrics_workspace_bytes(B, C, H, W))
    if nbytes < 0:
        check(nbytes)
    with torch.cuda.device(x.device):
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        out = torch.empty(B, 4, dtype=torch.float32, device=x.device)
        check(lib.rdg_image_metrics(ptr(x), ptr(y), B, C, H, W, value_range, ptr(out), ptr(ws), nbytes, _lib.stream_ptr()))
    return out


def masked_image_metrics(pred: torch.Tensor, gt: torch.Tensor, mask: torch.Tensor, value_range: float = 1.0) -> torch.Tensor:
    """(mmse, mpsnr, mssim) of every image pair over its covisibility mask, DyCheck's masked metrics (the iPhone protocol's
    mPSNR / mSSIM), as a [B, 3] float32 tensor on the inputs' device, without a host read.

    pred, gt as for image_metrics; mask: [1, H, W] for [C, H, W] inputs, [B, 1, H, W] for [B, C, H, W], shared by the
    channels; bool, uint8, half and double are converted to float32.  The mask is applied as a weight and not validated
    (DyCheck's masks are binary).  mmse = sum m (x - y)^2 / (C sum m), mpsnr = 10 log10(value_range^2 / mmse) without an
    epsilon; mssim is the mean over all C (H - 10) (W - 10) positions of the SSIM map of a masked (partial-convolution)
    Gaussian window, so a window without a covisible pixel counts as 1 and mssim is not the masked mean of image_metrics'
    SSIM map.  An empty mask gives (NaN, NaN, 1).  Values where the mask is 0 do not change a bit of the result (NaN and Inf
    included).  Not differentiable; an image's row does not depend on the rest of the batch, and repeated calls give
    identical bits."""
    x, y, value_range = _pair("masked_image_metrics", pred, gt, value_range)
    B, C, H, W = x.shape
    if not torch.is_tensor(mask):
        raise TypeError(f"masked_image_metrics: mask must be a tensor, got {type(mask).__name__}")
    if not mask.is_cuda:
        raise RuntimeError(f"masked_image_metrics: mask is on {mask.device}; rodygs_b200 runs on CUDA tensors only (no CPU fallback)")
    want = (B, 1, H, W) if pred.dim() == 4 else (1, H, W)
    if tuple(mask.shape) != want:
        raise ValueError(f"masked_image_metrics: mask must have shape {want} for pred of shape {tuple(pred.shape)}, "
                         f"got {tuple(mask.shape)}")
    if mask.device != x.device:
        raise ValueError(f"masked_image_metrics: mask is on {mask.device} but pred on {x.device}")
    m = mask.detach().to(torch.float32).reshape(B, H, W).contiguous()
    lib = _lib.load()
    nbytes = int(lib.rdg_masked_image_metrics_workspace_bytes(B, C, H, W))
    if nbytes < 0:
        check(nbytes)
    with torch.cuda.device(x.device):
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        out = torch.empty(B, 3, dtype=torch.float32, device=x.device)
        check(lib.rdg_masked_image_metrics(ptr(x), ptr(y), ptr(m), B, C, H, W, value_range, ptr(out), ptr(ws), nbytes,
                                           _lib.stream_ptr()))
    return out
