"""Time the drop-in KNN calls on the GPU with CUDA events after warm-up:

* simple_knn distCUDA2 at 120 K points (the initial cloud of configs/train/train_kubric_mrig.yaml:42,102), 1 M and 6 M,
  on a uniform cube and on a surface cloud (a floor and two walls: the grid aims at 2 points per cell by volume, so a
  2-D point set crowds the cells it crosses);
* pytorch3d knn_points forward + backward, self-query, K = 8, at 500 K points (the rigidity sample of BASELINE config 4).

Each call is repeated on the same input, so the points (16 B each after the counting sort) stay in L2 from the second
call on up to ~6 M points.  Prints the device name and power limit, then one JSON line per case.

    python tools/knn_bench.py [--iters 20] [--warmup 3] [--out knn_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def cloud(kind: str, n: int, gen: torch.Generator) -> torch.Tensor:
    if kind == "uniform":
        return torch.rand(n, 3, generator=gen) * 4 - 2
    uv = torch.rand(n, 2, generator=gen) * 4
    which = torch.randint(0, 3, (n,), generator=gen)
    z = torch.zeros(n)
    planes = torch.stack([torch.stack([uv[:, 0], uv[:, 1], z], 1), torch.stack([z, uv[:, 0], uv[:, 1]], 1),
                          torch.stack([uv[:, 0], z, uv[:, 1]], 1)])
    return planes[which, torch.arange(n)]


def time_ms(fn, iters: int, warmup: int):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return times[len(times) // 2], times[0]


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or "not measured"
    except (OSError, subprocess.SubprocessError):
        return "not measured"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("knn_bench needs a CUDA device (there is no CPU path to time)")
    from simple_knn._C import distCUDA2
    import pytorch3d.ops as torch3d

    head = {"device": torch.cuda.get_device_name(), "power_limit": power_limit()}
    print(json.dumps(head), flush=True)
    rows = []
    gen = torch.Generator().manual_seed(0)
    for kind in ("uniform", "surface"):
        for n in (120_000, 1_000_000, 6_000_000):
            p = cloud(kind, n, gen).cuda()
            med, best = time_ms(lambda: distCUDA2(p), args.iters, args.warmup)
            rows.append({"case": "distCUDA2", "cloud": kind, "n": n, "ms_median": round(med, 4), "ms_min": round(best, 4)})
            print(json.dumps(rows[-1]), flush=True)
    n, K = 500_000, 8
    p = cloud("uniform", n, gen).cuda().requires_grad_(True)
    w = torch.randn(1, n, K, device="cuda")

    def fwd_bwd():
        dists, _, _ = torch3d.knn_points(p[None], p[None], K=K)
        (dists * w).sum().backward()

    for name, fn in (("knn_points fwd", lambda: torch3d.knn_points(p[None], p[None], K=K)), ("knn_points fwd+bwd", fwd_bwd)):
        med, best = time_ms(fn, args.iters, args.warmup)
        rows.append({"case": name, "cloud": "uniform", "n": n, "K": K, "ms_median": round(med, 4), "ms_min": round(best, 4)})
        print(json.dumps(rows[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({**head, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
