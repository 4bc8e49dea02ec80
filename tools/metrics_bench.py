"""Time rdg_image_metrics (PSNR / SSIM / MS-SSIM, one pass per scale) against a float32 F.conv2d / F.avg_pool2d restatement
of the same definitions, and rdg_masked_image_metrics (mPSNR / mSSIM over a covisibility mask) against a float32 F.conv2d
restatement of its partial convolution, on the same device; print one JSON line for each, with the GPU's name and power
limit.

    python tools/metrics_bench.py [--batch 8] [--height 1080] [--width 1920] [--iters 50] [--warmup 5] [--out FILE]

Inputs are 8 seeded random pairs at 1920x1080 by default: 400 MB of input, more than the 126 MB L2, so every timed
pass reads its scale-0 input from HBM.  The masked kernel gets a seeded mask of smooth blobs with ragged edges and
single-pixel holes, about half the image covisible.  CUDA events around `iters` back-to-back calls after `warmup` calls of
each path."""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rodygs_b200 import _lib  # noqa: E402
from rodygs_b200._lib import check, ptr  # noqa: E402

HBM_BYTES_PER_S = 7.7e12      # HGX B200 data sheet, one GPU
MS_WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)


def torch_metrics(x, y, value_range=1.0):
    """The definitions restated with PyTorch ops in the inputs' dtype: [B, 4] (mse, psnr, ssim, ms_ssim)."""
    ch = x.shape[1]
    g = torch.exp(-((torch.arange(11, dtype=torch.float64) - 5) ** 2) / 4.5)
    taps = (g / g.sum()).to(dtype=x.dtype, device=x.device)
    C1, C2 = (0.01 * value_range) ** 2, (0.03 * value_range) ** 2

    def blur(t):
        t = F.conv2d(t, taps.view(1, 1, 1, -1).expand(ch, 1, 1, 11), groups=ch)
        return F.conv2d(t, taps.view(1, 1, -1, 1).expand(ch, 1, 11, 1), groups=ch)

    def ss_cs(a, b):
        ma, mb = blur(a), blur(b)
        saa, sbb, sab = blur(a * a) - ma * ma, blur(b * b) - mb * mb, blur(a * b) - ma * mb
        cs = (2 * sab + C2) / (saa + sbb + C2)
        return ((2 * ma * mb + C1) / (ma * ma + mb * mb + C1) * cs).mean((-1, -2)), cs.mean((-1, -2))

    mse = ((x - y) ** 2).mean((1, 2, 3))
    m = None
    for s in range(5):
        if s:
            x, y = F.avg_pool2d(x, 2, ceil_mode=True), F.avg_pool2d(y, 2, ceil_mode=True)
        ss, cs = ss_cs(x, y)
        if s == 0:
            ssim = ss.mean(1)
        term = (ss if s == 4 else cs).relu() ** MS_WEIGHTS[s]
        m = term if m is None else m * term
    return torch.stack([mse, 10 * torch.log10(value_range ** 2 / (mse + 1e-8)), ssim, m.mean(1)], 1)


def torch_masked_metrics(x, y, m, value_range=1.0):
    """The masked definitions restated with PyTorch ops in the inputs' dtype: [B, 3] (mmse, mpsnr, mssim); m [B, 1, H, W]."""
    B, ch, H, W = x.shape
    g = torch.exp(-((torch.arange(11, dtype=torch.float64) - 5) ** 2) / 4.5)
    taps = (g / g.sum()).to(dtype=x.dtype, device=x.device)
    ones = torch.ones(11, dtype=x.dtype, device=x.device)
    C1, C2 = (0.01 * value_range) ** 2, (0.03 * value_range) ** 2
    mb = m.expand(B, ch, H, W).reshape(B * ch, 1, H, W)
    n1 = F.conv2d(mb, ones.view(1, 1, 1, 11))
    v1 = (n1 != 0).to(x.dtype)
    n2 = F.conv2d(v1, ones.view(1, 1, 11, 1))

    def P(z):
        p1 = torch.where(n1 != 0, F.conv2d(mb * z.reshape(B * ch, 1, H, W), taps.view(1, 1, 1, 11)) * 11 / n1, 0.0)
        return torch.where(n2 != 0, F.conv2d(v1 * p1, taps.view(1, 1, 11, 1)) * 11 / n2, 0.0).view(B, ch, H - 10, W - 10)

    mx, my = P(x), P(y)
    sxx, syy = (P(x * x) - mx * mx).clamp(min=0), (P(y * y) - my * my).clamp(min=0)
    s = P(x * y) - mx * my
    sxy = torch.sign(s) * torch.minimum((sxx * syy).sqrt(), s.abs())
    ssim = ((2 * mx * my + C1) * (2 * sxy + C2) / ((mx * mx + my * my + C1) * (sxx + syy + C2))).mean((1, 2, 3))
    mse = (m * (x - y) ** 2).sum((1, 2, 3)) / (ch * m.sum((1, 2, 3)))
    return torch.stack([mse, 10 * torch.log10(value_range ** 2 / mse), ssim], 1)


def covisibility_mask(B, H, W, gen):
    low = torch.rand(B, 1, H // 40 + 2, W // 40 + 2, device="cuda", generator=gen)
    ragged = F.interpolate(low, size=(H, W), mode="bilinear", align_corners=False)
    ragged = ragged + 0.1 * torch.rand(B, 1, H, W, device="cuda", generator=gen)
    holes = torch.rand(B, 1, H, W, device="cuda", generator=gen) < 0.01
    return ((ragged > 0.55) & ~holes).float()


def algorithmic_bytes(B, C, H, W):
    """Scale 0 reads pred and gt once (8 B per pixel and channel); each coarser scale is written by the pass before it
    and read by its own pass (2 x 8 B per pooled pixel and channel).  The per-CTA partial sums are negligible."""
    total, h, w = B * C * H * W * 8, H, W
    for _ in range(4):
        h, w = (h + 1) // 2, (w + 1) // 2
        total += 2 * B * C * h * w * 8
    return total


def gpu_identity():
    idx = torch.cuda.current_device()
    try:
        q = subprocess.run(["nvidia-smi", f"--id={idx}", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (s.strip() for s in q.split(","))
    except Exception as e:   # noqa: BLE001 - the number is still reported, with what is known
        name, power = torch.cuda.get_device_name(idx), f"unknown ({type(e).__name__})"
    return name, power


def time_ms(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("metrics_bench: needs a CUDA device (times are measured on the GPU only)")
    torch.backends.cudnn.allow_tf32 = False          # both paths compute in float32
    B, Cc, H, W = args.batch, 3, args.height, args.width
    g = torch.Generator(device="cuda").manual_seed(0)
    pred = torch.rand(B, Cc, H, W, device="cuda", generator=g)
    gt = (0.7 * pred + 0.3 * torch.rand(B, Cc, H, W, device="cuda", generator=g)).contiguous()
    lib = _lib.load()
    nbytes = int(lib.rdg_image_metrics_workspace_bytes(B, Cc, H, W))
    if nbytes < 0:
        check(nbytes)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    out = torch.empty(B, 4, dtype=torch.float32, device="cuda")

    def kernel():
        check(lib.rdg_image_metrics(ptr(pred), ptr(gt), B, Cc, H, W, 1.0, ptr(out), ptr(ws), nbytes, _lib.stream_ptr()))

    launches0 = lib.rdg_launch_count()
    kernel()
    launches = lib.rdg_launch_count() - launches0
    ref = torch_metrics(pred, gt)
    torch.cuda.synchronize()
    diff = (out - ref).abs().max().item()
    k_ms = time_ms(kernel, args.iters, args.warmup)
    t_ms = time_ms(lambda: torch_metrics(pred, gt), max(5, args.iters // 5), 2)
    nb = algorithmic_bytes(B, Cc, H, W)
    name, power = gpu_identity()
    line = {"tool": "metrics_bench", "gpu": name, "power_limit": power, "batch": B, "height": H, "width": W,
            "kernel_launches_per_call": launches, "kernel_ms_per_image": round(k_ms / B, 4),
            "torch_f32_ms_per_image": round(t_ms / B, 4), "speedup": round(t_ms / k_ms, 2),
            "algorithmic_bytes_per_call": nb, "bytes_per_px_scale0": 8 * Cc,
            "achieved_GBps": round(nb / (k_ms * 1e-3) / 1e9, 1),
            "hbm_share": round(nb / (k_ms * 1e-3) / HBM_BYTES_PER_S, 3),
            "max_abs_diff_vs_torch_f32": diff, "cache": "inputs 2 x %.0f MB > 126 MB L2" % (pred.numel() * 4 / 1e6)}

    # masked: reads pred, gt (B C H W floats each) and the mask (B H W floats) once
    mask = covisibility_mask(B, H, W, g)
    mnbytes = int(lib.rdg_masked_image_metrics_workspace_bytes(B, Cc, H, W))
    if mnbytes < 0:
        check(mnbytes)
    mws = torch.empty(mnbytes, dtype=torch.uint8, device="cuda")
    mout = torch.empty(B, 3, dtype=torch.float32, device="cuda")

    def masked_kernel():
        check(lib.rdg_masked_image_metrics(ptr(pred), ptr(gt), ptr(mask), B, Cc, H, W, 1.0, ptr(mout), ptr(mws), mnbytes,
                                           _lib.stream_ptr()))

    launches0 = lib.rdg_launch_count()
    masked_kernel()
    mlaunches = lib.rdg_launch_count() - launches0
    mref = torch_masked_metrics(pred, gt, mask)
    torch.cuda.synchronize()
    mdiff = (mout - mref).abs().max().item()
    mk_ms = time_ms(masked_kernel, args.iters, args.warmup)
    mt_ms = time_ms(lambda: torch_masked_metrics(pred, gt, mask), max(5, args.iters // 5), 2)
    mnb = B * Cc * H * W * 8 + B * H * W * 4
    mline = {"tool": "metrics_bench_masked", "gpu": name, "power_limit": power, "batch": B, "height": H, "width": W,
             "covisible_fraction": round(mask.mean().item(), 3), "kernel_launches_per_call": mlaunches,
             "kernel_ms_per_image": round(mk_ms / B, 4), "torch_f32_ms_per_image": round(mt_ms / B, 4),
             "speedup": round(mt_ms / mk_ms, 2), "algorithmic_bytes_per_call": mnb,
             "achieved_GBps": round(mnb / (mk_ms * 1e-3) / 1e9, 1),
             "hbm_share": round(mnb / (mk_ms * 1e-3) / HBM_BYTES_PER_S, 3),
             "max_abs_diff_vs_torch_f32": mdiff, "cache": line["cache"]}
    lines = [json.dumps(line), json.dumps(mline)]
    print("\n".join(lines))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    for what, d in (("kernel", diff), ("masked kernel", mdiff)):
        if not math.isfinite(d) or d > 1e-3:
            raise SystemExit(f"metrics_bench: {what} and PyTorch restatement disagree by {d}")


if __name__ == "__main__":
    main()
