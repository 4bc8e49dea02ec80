"""Exporting the BASELINE config-5 scene (6 M Gaussians, 50 % dynamic, T = 100, SH degree 3) at one time t as a 3DGS PLY
file, in one call:

* kernel: SplatTrainStep.export_3dgs (one rdg_export_3dgs launch), CUDA events, after a warm-up; median of --runs;
* copy:   the records [N, 62] device -> pinned host (Tensor.copy_), CUDA events;
* write:  rodygs_b200.ply.write_ply of the host records to a temporary file that is deleted afterwards (host clock, the
          file flushed with os.fsync), a number about that machine's disk, not the GPU.

The scene (about 1.8 GB of parameters) is far larger than the L2.  Prints one JSON line with the device name and power limit.
Usage: python tools/export_bench.py [--runs R] [--out file.json]"""
import argparse
import json
import os
import statistics
import sys
import tempfile
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rodygs_b200 import ply, synthetic  # noqa: E402
from rodygs_b200.trainer import SplatTrainStep  # noqa: E402
from camera_bench import gpu_identity  # noqa: E402
from render_bench import timed_ms  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--writes", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    N, H, W, T, _ = synthetic.CONFIGS["c5_infer"]
    scene = synthetic.to_device(synthetic.make_scene(N, H, W, T, seed=0), "cuda")
    step = SplatTrainStep(scene, H, W, sh_degree=3, w_pearson=0.0)
    del scene
    bt = step.p("table")[T // 2].clone()
    out = {}

    def export():
        out["rec"] = step.export_3dgs(bt)

    for _ in range(3):
        export()
    host = torch.empty(out["rec"].shape, dtype=torch.float32, pin_memory=True)

    def copy():
        host.copy_(out["rec"], non_blocking=True)

    copy()
    kernel, d2h = [], []
    for _ in range(args.runs):
        kernel.append(timed_ms(export))
        d2h.append(timed_ms(copy))
    write = []
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "scene.ply")
        for _ in range(args.writes):
            t0 = time.perf_counter()
            ply.write_ply(path, host.numpy())
            with open(path, "rb+") as f:
                os.fsync(f.fileno())
            write.append(1e3 * (time.perf_counter() - t0))
            size = os.path.getsize(path)
            os.remove(path)
    n = step.ns + step.nd
    name, power = gpu_identity()
    med = statistics.median
    res = {"tool": "export_bench", "device": name, "power_limit": power, "workload": "c5_infer", "n": n,
           "n_dynamic": step.nd, "num_times": T, "sh_degree": 3, "runs": args.runs, "record_bytes": 248,
           "records_bytes": 248 * n, "file_bytes": size,
           "kernel_ms": {"median": med(kernel), "min": min(kernel), "max": max(kernel)},
           "copy_d2h_pinned_ms": {"median": med(d2h), "min": min(d2h), "max": max(d2h)},
           "write_ms_this_machines_disk": {"median": med(write), "min": min(write), "max": max(write), "writes": args.writes},
           "kernel_GBps_records_written": 248 * n / (med(kernel) * 1e6)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
