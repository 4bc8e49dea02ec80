"""Time rdg_lpips (AlexNet and VGG-16 LPIPS, convolutions on tcgen05 tensor cores in TF32) per image pair, its conv
kernel per layer, and a float32 F.conv2d restatement of the same definition with cuDNN's TF32 allowed (the reference's
arithmetic) and disallowed; in the same run, rdg_masked_lpips (mLPIPS) of the same pair under a seeded covisibility mask,
alternating with rdg_lpips call by call.  Prints one JSON line per backbone with the GPU's name, power limit and SM clock.

    python tools/lpips_bench.py [--height 1080] [--width 1920] [--iters 100] [--warmup 20] [--out FILE]

Weights are seeded random ones under the real key names (nothing is downloaded; the time does not depend on the values).
One seeded render-like pair at 1920x1080.  Per-pair times: CUDA events around each of `iters` calls after `warmup` calls,
reported as median / p10 / p90; rdg_lpips and rdg_masked_lpips are timed alternately in one loop, so both see the same
clocks.  The masked path's own kernels (the spatial pass and its finalize) are also timed from a torch.profiler run.  Per-layer conv times: device time of each lpips_conv_kernel launch from a torch.profiler
run of its own, median over 20 pairs.  Achieved TFLOP/s = 2 MAC / time, set against the data-sheet dense TF32 rate of
one HGX B200 GPU (1,125 TFLOP/s; a data-sheet figure, not one measured here).  The VGG pair's activations (1.06 GB for
relu1_2 of the pair) exceed the 126 MB L2."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rodygs_b200.metrics import LPIPS_CONVS, LPIPS_TAPS, load_lpips, lpips, masked_lpips  # noqa: E402

TF32_DATASHEET_TFLOPS = 1125.0
POOLS = {"alex": {3: 3, 6: 3}, "vgg": {5: 2, 10: 2, 17: 2, 24: 2}}   # features.{i} -> kernel of the stride-2 pool before it
GEOM = {"alex": {0: (4, 2), 3: (1, 2)}}                               # (stride, padding) where not (1, 1)
TAPS = {"alex": (0, 3, 6, 8, 10), "vgg": (2, 7, 14, 21, 28)}


def weights(net, seed):
    g = torch.Generator().manual_seed(seed)
    bb = {}
    for i, cout, cin, k in LPIPS_CONVS[net]:
        bb[f"features.{i}.weight"] = torch.randn(cout, cin, k, k, generator=g) * (2.0 / (cin * k * k)) ** 0.5
        bb[f"features.{i}.bias"] = torch.randn(cout, generator=g) * 0.01
    lin = {f"lin{l}.model.1.weight": torch.rand(1, c, 1, 1, generator=g) * 0.2 for l, c in enumerate(LPIPS_TAPS[net])}
    return bb, lin


def layer_shapes(net, H, W):
    """[(features index, Cout, Cin, k, stride, pad, H_in, W_in, H_out, W_out)] of the convs."""
    out, h, w = [], H, W
    for i, cout, cin, k in LPIPS_CONVS[net]:
        if i in POOLS[net]:
            pk = POOLS[net][i]
            h, w = (h - pk) // 2 + 1, (w - pk) // 2 + 1
        s, p = GEOM.get(net, {}).get(i, (1, 1))
        ho, wo = (h + 2 * p - k) // s + 1, (w + 2 * p - k) // s + 1
        out.append((i, cout, cin, k, s, p, h, w, ho, wo))
        h, w = ho, wo
    return out


def torch_lpips(pred, gt, net, dev_w):
    """The definition restated with F.conv2d / F.max_pool2d in float32: [B]."""
    mu = torch.tensor([0.485, 0.456, 0.406], device=pred.device).view(1, 3, 1, 1)
    sd = torch.tensor([0.229, 0.224, 0.225], device=pred.device).view(1, 3, 1, 1)
    z = (torch.cat([pred, gt]) - mu) / sd
    B, total, t = pred.shape[0], 0.0, 0
    for i, _, _, _ in LPIPS_CONVS[net]:
        if i in POOLS[net]:
            z = F.max_pool2d(z, POOLS[net][i], 2)
        s, p = GEOM.get(net, {}).get(i, (1, 1))
        z = F.relu(F.conv2d(z, dev_w[f"features.{i}.weight"], dev_w[f"features.{i}.bias"], stride=s, padding=p))
        if i in TAPS[net]:
            n = z / (z.pow(2).sum(1, keepdim=True).sqrt() + 1e-10)
            total = total + (dev_w[f"lin{t}.model.1.weight"] * (n[:B] - n[B:]) ** 2).sum(1).mean((1, 2))
            t += 1
    return total


def gpu_identity():
    idx = torch.cuda.current_device()
    try:
        q = subprocess.run(["nvidia-smi", f"--id={idx}", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, sm, sm_max = (s.strip() for s in q.split(","))
    except Exception as e:   # noqa: BLE001 - the number is still reported, with what is known
        name, power, sm, sm_max = torch.cuda.get_device_name(idx), f"unknown ({type(e).__name__})", "unknown", "unknown"
    return {"gpu": name, "power_limit": power, "sm_clock_at_query": sm, "sm_clock_max": sm_max}


def _summary(ts):
    ts = sorted(ts)
    q = lambda f: ts[min(len(ts) - 1, int(f * len(ts)))]   # noqa: E731
    return {"median": round(statistics.median(ts), 4), "p10": round(q(0.1), 4), "p90": round(q(0.9), 4)}


def event_times(fn, iters, warmup):
    return alternating_event_times([fn], iters, warmup)[0]


def alternating_event_times(fns, iters, warmup):
    """CUDA-event times of each of fns, called in turn `iters` times after `warmup` rounds."""
    for _ in range(warmup):
        for fn in fns:
            fn()
    torch.cuda.synchronize()
    ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in fns] for _ in range(iters)]
    for row in ev:
        for fn, (a, b) in zip(fns, row):
            a.record()
            fn()
            b.record()
    torch.cuda.synchronize()
    return [_summary([row[k][0].elapsed_time(row[k][1]) for row in ev]) for k in range(len(fns))]


def covisibility_mask(H, W, g):
    """[1, 1, H, W]: blobs with ragged edges and single-pixel holes, about half the image covisible."""
    low = torch.rand(1, 1, H // 40 + 2, W // 40 + 2, device="cuda", generator=g)
    smooth = F.interpolate(low, size=(H, W), mode="bilinear", align_corners=False)
    ragged = smooth + 0.1 * torch.rand(1, 1, H, W, device="cuda", generator=g)
    holes = torch.rand(1, 1, H, W, device="cuda", generator=g) < 0.01
    return ((ragged > 0.55) & ~holes).float()


def conv_layer_ms(fn, nconv, pairs=20):
    """Median device time of each lpips_conv_kernel launch, by layer, from a profiler run of `pairs` calls."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(pairs):
            fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if "lpips_conv_kernel" in e.name]
    ev.sort(key=lambda e: e.time_range.start)
    assert len(ev) == pairs * nconv, (len(ev), pairs, nconv)
    return [statistics.median(ev[p * nconv + l].time_range.elapsed_us() for p in range(pairs)) / 1e3 for l in range(nconv)]


def kernels_ms(fn, names, pairs=20):
    """Median device time per pair of the launches whose kernel name holds one of `names`, from a profiler run."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(pairs):
            fn()
        torch.cuda.synchronize()
    out = {}
    for name in names:
        ev = sorted((e for e in prof.events() if name in e.name), key=lambda e: e.time_range.start)
        assert len(ev) == pairs, (name, len(ev), pairs)
        out[name] = round(statistics.median(e.time_range.elapsed_us() for e in ev) / 1e3, 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lpips_bench: needs a CUDA device (there is no CPU path to time)")
    H, W = args.height, args.width
    g = torch.Generator(device="cuda").manual_seed(0)
    low = torch.rand(1, 3, H // 60 + 2, W // 60 + 2, device="cuda", generator=g)
    pred = F.interpolate(low, size=(H, W), mode="bilinear", align_corners=False)
    gt = (pred + 0.05 * torch.randn(pred.shape, device="cuda", generator=g)).clamp(0, 1)
    mask = covisibility_mask(H, W, torch.Generator(device="cuda").manual_seed(1))
    ident = gpu_identity()
    lines = []
    saved = torch.backends.cudnn.allow_tf32
    for k, net in enumerate(("alex", "vgg")):
        bb, lin = weights(net, k)
        w = load_lpips(net, bb, lin)
        dev_w = {key: v.cuda() for key, v in {**bb, **lin}.items()}
        shapes = layer_shapes(net, H, W)
        macs = [2 * ho * wo * cout * cin * kk * kk for (_, cout, cin, kk, _, _, _, _, ho, wo) in shapes]
        kern, mkern = alternating_event_times([lambda: lpips(pred, gt, w), lambda: masked_lpips(pred, gt, mask, w)],
                                              args.iters, args.warmup)
        per_layer = conv_layer_ms(lambda: lpips(pred, gt, w), len(shapes))
        masked_own = kernels_ms(lambda: masked_lpips(pred, gt, mask, w),
                                ("lpips_spatial_kernel", "lpips_masked_finalize_kernel"))
        res = {}
        for tf32 in (True, False):
            torch.backends.cudnn.allow_tf32 = tf32
            with torch.no_grad():
                res[tf32] = event_times(lambda: torch_lpips(pred, gt, net, dev_w), args.iters, args.warmup)
                ref = torch_lpips(pred, gt, net, dev_w)
            # cuDNN per layer on the same shapes
            cud = []
            for (i, cout, cin, kk, s, p, h, ww, _, _) in shapes:
                x = torch.rand(2, cin, h, ww, device="cuda", generator=g)
                wt, bi = dev_w[f"features.{i}.weight"], dev_w[f"features.{i}.bias"]
                with torch.no_grad():
                    cud.append(event_times(lambda: F.relu(F.conv2d(x, wt, bi, stride=s, padding=p)), 20, 5)["median"])
                del x
            res[f"layers_{tf32}"] = cud
            res[f"value_{tf32}"] = ref.item()
        torch.backends.cudnn.allow_tf32 = saved
        got = lpips(pred, gt, w).item()
        got_masked = masked_lpips(pred, gt, mask, w).item()
        layers = []
        for (i, cout, cin, kk, s, p, h, ww, ho, wo), mac, ms, ctf, cfp in zip(shapes, macs, per_layer, res["layers_True"],
                                                                               res["layers_False"]):
            layers.append({"layer": f"features.{i}", "cin": cin, "cout": cout, "k": kk, "out": [ho, wo],
                           "gmac_pair": round(mac / 1e9, 2), "kernel_ms": round(ms, 4),
                           "kernel_tflops": round(2 * mac / (ms * 1e-3) / 1e12, 1),
                           "share_of_datasheet_tf32": round(2 * mac / (ms * 1e-3) / 1e12 / TF32_DATASHEET_TFLOPS, 3),
                           "cudnn_tf32_ms": ctf, "cudnn_fp32_ms": cfp})
        total_mac = sum(macs)
        line = {"tool": "lpips_bench", **ident, "net": net, "height": H, "width": W, "pairs_per_call": 1,
                "iters": args.iters, "warmup": args.warmup, "gmac_pair": round(total_mac / 1e9, 1),
                "kernel_ms_per_pair": kern, "cudnn_tf32_ms_per_pair": res[True], "cudnn_fp32_ms_per_pair": res[False],
                "kernel_tflops_whole_pair": round(2 * total_mac / (kern["median"] * 1e-3) / 1e12, 1),
                "datasheet_dense_tf32_tflops": TF32_DATASHEET_TFLOPS, "layers": layers,
                "value_kernel": got, "value_cudnn_tf32": res["value_True"], "value_cudnn_fp32": res["value_False"],
                "mask_covisible": round(mask.mean().item(), 4), "masked_kernel_ms_per_pair": mkern,
                "masked_minus_plain_ms_median": round(mkern["median"] - kern["median"], 4),
                "masked_own_kernels_ms": masked_own, "value_masked_kernel": got_masked}
        lines.append(json.dumps(line))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
