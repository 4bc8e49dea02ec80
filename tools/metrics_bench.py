"""Time rdg_image_metrics (PSNR / SSIM / MS-SSIM, one pass per scale) against a float32 F.conv2d / F.avg_pool2d restatement
of the same definitions on the same device, and print one JSON line with the GPU's name and power limit.

    python tools/metrics_bench.py [--batch 8] [--height 1080] [--width 1920] [--iters 50] [--warmup 5] [--out FILE]

Inputs are 8 seeded random pairs at 1920x1080 by default: 400 MB of input, more than the 126 MB L2, so every timed
pass reads its scale-0 input from HBM.  CUDA events around `iters` back-to-back calls after `warmup` calls of each path."""
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
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")
    if not math.isfinite(diff) or diff > 1e-3:
        raise SystemExit(f"metrics_bench: kernel and PyTorch restatement disagree by {diff}")


if __name__ == "__main__":
    main()
