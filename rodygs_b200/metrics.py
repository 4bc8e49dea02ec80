"""Evaluation image metrics on the device: MSE, PSNR, SSIM and MS-SSIM in one fused pass per scale (rdg_image_metrics),
their masked forms over a covisibility mask, mPSNR and mSSIM (rdg_masked_image_metrics), LPIPS (rdg_lpips) and its masked
form, mLPIPS (rdg_masked_lpips); and the trajectory errors ATE / RPE of learned cameras (trajectory_errors, float64 torch).

These are the metrics the reference reports for held-out views (RoDyGSEvaluator.eval, VizScoreEvaluator, through piqa):
an 11x11 Gaussian window (sigma 1.5) over the VALID region only, averaged per channel, and MS-SSIM over five scales.  They
are not the training SSIM in SplatTrainStep.loss_parts[2], which zero-pads the window over the full image and gives a
lower number near the borders.  piqa's conventions are recalled, not pinned against piqa itself: INTEGRATION.md,
"Scoring held-out views", states them.
"""
from __future__ import annotations

import ctypes

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
    _mask_shape("masked_image_metrics", mask, pred)
    m = _mask_on("masked_image_metrics", mask, x)
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


def _mask_shape(fn: str, mask: torch.Tensor, pred: torch.Tensor):
    """mask must be [1, H, W] for pred [C, H, W] and [B, 1, H, W] for pred [B, C, H, W]."""
    H, W = pred.shape[-2:]
    want = (pred.shape[0], 1, H, W) if pred.dim() == 4 else (1, H, W)
    if tuple(mask.shape) != want:
        raise ValueError(f"{fn}: mask must have shape {want} for pred of shape {tuple(pred.shape)}, got {tuple(mask.shape)}")


def _mask_on(fn: str, mask: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """The checked mask on x's device as contiguous float32 [B, H, W]."""
    if mask.device != x.device:
        raise ValueError(f"{fn}: mask is on {mask.device} but pred on {x.device}")
    B, _, H, W = x.shape
    return mask.detach().to(torch.float32).reshape(B, H, W).contiguous()


# ---- LPIPS ---------------------------------------------------------------------------------------------------------------

# features.{i} of each torchvision backbone that is a conv, in network order, with (Cout, Cin, k); the taps' channels
LPIPS_CONVS = {
    "alex": [(0, 64, 3, 11), (3, 192, 64, 5), (6, 384, 192, 3), (8, 256, 384, 3), (10, 256, 256, 3)],
    "vgg": [(0, 64, 3, 3), (2, 64, 64, 3), (5, 128, 64, 3), (7, 128, 128, 3), (10, 256, 128, 3), (12, 256, 256, 3),
            (14, 256, 256, 3), (17, 512, 256, 3), (19, 512, 512, 3), (21, 512, 512, 3), (24, 512, 512, 3),
            (26, 512, 512, 3), (28, 512, 512, 3)],
}
LPIPS_TAPS = {"alex": (64, 192, 384, 256, 256), "vgg": (64, 128, 256, 512, 512)}
_LPIPS_NET = {"alex": 0, "vgg": 1}                 # RDG_LPIPS_ALEX, RDG_LPIPS_VGG
_LPIPS_MIN_EDGE = {"alex": 31, "vgg": 16}         # the last tap is not empty


class LpipsWeights:
    """One backbone's weights packed on the device for rodygs_b200.metrics.lpips (built by load_lpips)."""

    def __init__(self, net: str, packed: torch.Tensor):
        self.net = net
        self.packed = packed

    def __repr__(self):
        return f"LpipsWeights(net={self.net!r}, device={self.packed.device})"


def _state_dict(fn: str, what: str, src):
    if isinstance(src, dict):
        return src
    sd = torch.load(src, map_location="cpu", weights_only=True)
    if not isinstance(sd, dict):
        raise ValueError(f"{fn}: {what} {src!r} does not hold a state dict")
    return sd


def _tensor(fn: str, sd: dict, key: str, shape) -> torch.Tensor:
    if key not in sd:
        raise ValueError(f"{fn}: missing key {key!r}")
    t = sd[key]
    if not torch.is_tensor(t) or tuple(t.shape) != tuple(shape):
        got = tuple(t.shape) if torch.is_tensor(t) else type(t).__name__
        raise ValueError(f"{fn}: {key!r} must have shape {tuple(shape)}, got {got}")
    return t


def load_lpips(net: str, backbone, linear, device="cuda") -> LpipsWeights:
    """LPIPS weights of `net` ("alex" or "vgg") from the files a run of the reference already has; nothing is downloaded.

    backbone: the torchvision state dict of the backbone (e.g. alexnet-owt-7be5be79.pth, vgg16-397923af.pth) or its path;
    the keys read are features.{i}.weight / .bias of the convs (LPIPS_CONVS), classifier.* is ignored.  linear: the lpips
    package's heads (weights/v0.1/alex.pth, vgg.pth) or its path, keys lin{0..4}.model.1.weight [1, C_l, 1, 1].  Paths are
    read with torch.load(map_location="cpu", weights_only=True).  A missing key or a wrong shape raises ValueError naming
    the key.  Returns the weights packed for the conv kernels on `device` (one rdg_lpips_pack call)."""
    fn = "load_lpips"
    if net not in LPIPS_CONVS:
        raise ValueError(f"{fn}: net must be 'alex' or 'vgg', got {net!r}")
    bb, lin = _state_dict(fn, "backbone", backbone), _state_dict(fn, "linear", linear)
    ws, bs = [], []
    for i, cout, cin, k in LPIPS_CONVS[net]:
        ws.append(_tensor(fn, bb, f"features.{i}.weight", (cout, cin, k, k)))
        bs.append(_tensor(fn, bb, f"features.{i}.bias", (cout,)))
    ls = [_tensor(fn, lin, f"lin{l}.model.1.weight", (1, c, 1, 1)) for l, c in enumerate(LPIPS_TAPS[net])]
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(f"{fn}: device is {dev}; rodygs_b200 runs on CUDA tensors only (no CPU fallback)")
    ws, bs, ls = ([t.detach().to(device=dev, dtype=torch.float32).contiguous() for t in ts] for ts in (ws, bs, ls))
    lib = _lib.load()
    code = _LPIPS_NET[net]
    n = int(lib.rdg_lpips_packed_floats(code))
    arr = lambda ts: (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])   # noqa: E731
    with torch.cuda.device(dev):
        packed = torch.empty(n, dtype=torch.float32, device=dev)
        check(lib.rdg_lpips_pack(code, arr(ws), arr(bs), arr(ls), ptr(packed), n, _lib.stream_ptr()))
    return LpipsWeights(net, packed)


def _lpips_shapes(fn: str, pred, gt, weights):
    """The checks of lpips / masked_lpips that need no device: the weights' type, 3 channels, the backbone's least size."""
    if not isinstance(weights, LpipsWeights):
        raise TypeError(f"{fn}: weights must be an LpipsWeights from load_lpips, got {type(weights).__name__}")
    for name, t in (("pred", pred), ("gt", gt)):
        if torch.is_tensor(t) and t.dim() in (3, 4):
            if t.shape[-3] != 3:
                raise ValueError(f"{fn}: {name} must have 3 channels, got shape {tuple(t.shape)}")
            edge = _LPIPS_MIN_EDGE[weights.net]
            if min(t.shape[-2:]) < edge:
                raise ValueError(f"{fn}: {name} is {t.shape[-2]}x{t.shape[-1]}; the {weights.net} backbone needs H and W "
                                 f">= {edge}")


def lpips(pred: torch.Tensor, gt: torch.Tensor, weights: LpipsWeights, value_range: float = 1.0) -> torch.Tensor:
    """LPIPS (the lpips package v0.1, lpips=True, spatial=False) of every image pair as a [B] float32 tensor on the inputs'
    device, without a host read.

    pred, gt: [3, H, W] or [B, 3, H, W] CUDA tensors of the same shape in [0, value_range]; other dtypes are converted to
    float32.  H, W >= 31 for alex and >= 16 for vgg.  weights: from load_lpips, on the inputs' device.  The convolutions
    run on tensor cores in TF32 (the reference's arithmetic under cuDNN's default).  Not differentiable.  The result of a
    pair does not depend on the other pairs, and repeated calls give identical bits."""
    _lpips_shapes("lpips", pred, gt, weights)
    x, y, value_range = _pair("lpips", pred, gt, value_range)
    B, Cc, H, W = x.shape
    if weights.packed.device != x.device:
        raise ValueError(f"lpips: weights are on {weights.packed.device} but pred on {x.device}")
    lib = _lib.load()
    code = _LPIPS_NET[weights.net]
    nbytes = int(lib.rdg_lpips_workspace_bytes(code, H, W))
    if nbytes < 0:
        check(nbytes)
    with torch.cuda.device(x.device):
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        out = torch.empty(B, dtype=torch.float32, device=x.device)
        check(lib.rdg_lpips(ptr(x), ptr(y), B, Cc, H, W, value_range, code, ptr(weights.packed), weights.packed.numel(),
                            ptr(out), ptr(ws), nbytes, _lib.stream_ptr()))
    return out


def masked_lpips(pred: torch.Tensor, gt: torch.Tensor, mask: torch.Tensor, weights: LpipsWeights,
                 value_range: float = 1.0) -> torch.Tensor:
    """Masked LPIPS over a covisibility mask, DyCheck's mLPIPS (the iPhone protocol; DyCheck uses alex), of every image pair
    as a [B] float32 tensor on the inputs' device, without a host read.

    pred, gt, weights and value_range as for lpips; mask as for masked_image_metrics ([1, H, W] or [B, 1, H, W], shared by
    the channels; bool, uint8, half and double converted to float32; applied as a weight, not validated).  Both images are
    masked first (x_m = m x where m != 0, else 0), the lpips head of every tap position is upsampled bilinearly
    (align_corners=False) to H x W and summed over the taps, and the result is sum m map / sum m.  An empty mask gives NaN;
    values where the mask is 0 change no bit of the result (NaN and Inf included).  With an all-ones mask this equals lpips
    only where every tap size divides the image size (vgg at 64x64): bilinear upsampling of a 15x15 alex tap to 64x64 does
    not keep its mean.  Not differentiable.  The result of a pair does not depend on the other pairs, and repeated calls
    give identical bits."""
    fn = "masked_lpips"
    _lpips_shapes(fn, pred, gt, weights)
    if not torch.is_tensor(mask):
        raise TypeError(f"{fn}: mask must be a tensor, got {type(mask).__name__}")
    if torch.is_tensor(pred) and pred.dim() in (3, 4):
        _mask_shape(fn, mask, pred)
    x, y, value_range = _pair(fn, pred, gt, value_range)
    if not mask.is_cuda:
        raise RuntimeError(f"{fn}: mask is on {mask.device}; rodygs_b200 runs on CUDA tensors only (no CPU fallback)")
    m = _mask_on(fn, mask, x)
    B, Cc, H, W = x.shape
    if weights.packed.device != x.device:
        raise ValueError(f"{fn}: weights are on {weights.packed.device} but pred on {x.device}")
    lib = _lib.load()
    code = _LPIPS_NET[weights.net]
    nbytes = int(lib.rdg_masked_lpips_workspace_bytes(code, H, W))
    if nbytes < 0:
        check(nbytes)
    with torch.cuda.device(x.device):
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        out = torch.empty(B, dtype=torch.float32, device=x.device)
        check(lib.rdg_masked_lpips(ptr(x), ptr(y), ptr(m), B, Cc, H, W, value_range, code, ptr(weights.packed),
                                   weights.packed.numel(), ptr(out), ptr(ws), nbytes, _lib.stream_ptr()))
    return out


def trajectory_errors(pred_c2w: torch.Tensor, gt_c2w: torch.Tensor):
    """(ate, rpe_trans, rpe_rot_deg) of a learned camera trajectory, three float64 scalars on the inputs' device (no host
    read).  pred_c2w / gt_c2w: [C, 4, 4] camera-to-world matrices (mathematical row-major layout, C >= 2), in the same order.

    The predicted camera centres are aligned to the ground-truth ones by the Umeyama Sim(3) (rotation, translation and
    scale); ATE is the RMSE of the aligned centres.  The aligned predicted poses (R pred_R, s R pred_t + t) then give RPE over
    consecutive pairs: rel = inv(inv(gt_i) gt_{i+1}) (inv(pred_i) pred_{i+1}), rpe_trans the mean of |rel[:3, 3]|, rpe_rot_deg
    the mean of arccos(clamp((tr rel[:3, :3] - 1) / 2, -1, 1)) in degrees.  These are the compute_ATE / compute_rpe
    conventions of Nope-NeRF / CF-3DGS as recalled, not pinned (INTEGRATION.md "Learning the training cameras").  Computed
    in float64 with torch: C is at most a few thousand 4x4 matrices."""
    if not (torch.is_tensor(pred_c2w) and torch.is_tensor(gt_c2w) and pred_c2w.dim() == 3 and pred_c2w.shape[0] >= 2
            and tuple(pred_c2w.shape[1:]) == (4, 4) and pred_c2w.shape == gt_c2w.shape and pred_c2w.device == gt_c2w.device):
        got = [tuple(t.shape) if torch.is_tensor(t) else type(t).__name__ for t in (pred_c2w, gt_c2w)]
        raise ValueError(f"trajectory_errors: pred_c2w and gt_c2w must be [C, 4, 4] tensors on one device with C >= 2, got {got}")
    pred, gt = pred_c2w.double(), gt_c2w.double()
    n = pred.shape[0]
    # Umeyama: gt_centre ~ s R pred_centre + t
    x, y = pred[:, :3, 3], gt[:, :3, 3]
    mx, my = x.mean(0), y.mean(0)
    xc, yc = x - mx, y - my
    U, D, Vh = torch.linalg.svd(yc.t() @ xc / n)
    S = torch.ones(3, dtype=torch.float64, device=pred.device)
    S[2] = torch.where(torch.linalg.det(U) * torch.linalg.det(Vh) < 0, -1.0, 1.0)
    R = U @ torch.diag(S) @ Vh
    s = (D * S).sum() / ((xc * xc).sum() / n)
    t = my - s * (R @ mx)
    aligned = pred.clone()
    aligned[:, :3, :3] = R @ pred[:, :3, :3]
    aligned[:, :3, 3] = s * x @ R.t() + t
    ate = ((aligned[:, :3, 3] - y) ** 2).sum(-1).mean().sqrt()
    inv_gt, inv_pred = torch.linalg.inv(gt), torch.linalg.inv(aligned)
    rel = torch.linalg.inv(inv_gt[:-1] @ gt[1:]) @ (inv_pred[:-1] @ aligned[1:])
    rpe_trans = rel[:, :3, 3].norm(dim=-1).mean()
    # the arccos of the definition as atan2(sin, cos): the same angle for a rotation, but without arccos' loss of precision
    # near 0 (arccos(1 - 1e-16) is already 1.4e-8)
    cos = ((rel[:, 0, 0] + rel[:, 1, 1] + rel[:, 2, 2] - 1.0) / 2.0).clamp(-1.0, 1.0)
    sin = torch.stack([rel[:, 2, 1] - rel[:, 1, 2], rel[:, 0, 2] - rel[:, 2, 0], rel[:, 1, 0] - rel[:, 0, 1]], -1).norm(dim=-1) / 2.0
    rpe_rot = torch.rad2deg(torch.atan2(sin, cos)).mean()
    return ate, rpe_trans, rpe_rot


def pck(pred: torch.Tensor, gt: torch.Tensor, visible: torch.Tensor, height: int, width: int, ratio: float = 0.05):
    """PCK-T (percentage of correct keypoint transfers), [B] float64 on the inputs' device (no host read): for each row b
    the fraction of the points with visible[b] != 0 whose prediction lies strictly within ratio * max(height, width) pixels
    of the ground truth, |pred - gt|_2 < ratio * max(H, W).  pred / gt [B, P, 2] pixel coordinates, visible [B, P] (bool or
    numbers).  A NaN prediction counts as wrong; a row without a visible point is NaN.

    DyCheck's keypoint-transfer protocol, as recalled and not pinned (INTEGRATION.md §10): a ratio of 0.05 of the longer
    side, pairs of training frames, keypoints counted where they are visible in both frames; the caller converts DyCheck's
    keypoint pixel convention to the rasterizer's (pixel (x, y) centred at integer x, y) before tracking.  Computed in
    float64 with torch, as trajectory_errors: B x P is at most a few thousand points."""
    if not (torch.is_tensor(pred) and torch.is_tensor(gt) and torch.is_tensor(visible) and pred.dim() == 3
            and pred.shape[-1] == 2 and pred.shape == gt.shape and tuple(visible.shape) == tuple(pred.shape[:2])
            and pred.device == gt.device == visible.device):
        got = [f"{tuple(t.shape)} {t.device}" if torch.is_tensor(t) else type(t).__name__ for t in (pred, gt, visible)]
        raise ValueError(f"pck: pred and gt must be [B, P, 2] and visible [B, P] tensors on one device, got {got}")
    if not (int(height) > 0 and int(width) > 0 and ratio > 0):
        raise ValueError(f"pck: height, width and ratio must be positive, got {height}, {width}, {ratio}")
    vis = visible != 0
    dist = torch.linalg.vector_norm(pred.double() - gt.double(), dim=-1)
    correct = (dist < ratio * max(int(height), int(width))) & vis        # NaN < x is False: a NaN prediction is wrong
    return correct.sum(-1).double() / vis.sum(-1).double()                 # 0 / 0 = NaN: no visible point
