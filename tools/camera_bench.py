"""Cost of learning the training cameras, with CUDA events:

* SplatTrainStep.camera_step (rdg_camera_grad + the all-reduce, a no-op on one process + rdg_camera_adam + the one host read
  of the index error word) at C = 100 and C = 2000 cameras with one collected view, and the two kernels alone;
* the BASELINE config-4 training step (2 M Gaussians at 1920x1080, forward_backward) without camera learning against the same
  step with forward_backward(camera=c) + camera_step, alternating run by run.

Prints one JSON line with the device name and power limit.  Usage: python tools/camera_bench.py [--out file.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rodygs_b200 import _lib, synthetic  # noqa: E402
from rodygs_b200.optim import CameraLRs  # noqa: E402
from rodygs_b200.trainer import SplatTrainStep  # noqa: E402


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}", "--query-gpu=name,power.limit",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (s.strip() for s in q.split(","))
    except Exception as e:   # noqa: BLE001 - the numbers are still reported, with what is known
        name, power = torch.cuda.get_device_name(), f"unknown ({type(e).__name__})"
    return name, power


def timed_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def random_viewmats(C, seed):
    g = torch.Generator().manual_seed(seed)
    q = torch.nn.functional.normalize(torch.randn(C, 4, generator=g, dtype=torch.float64), dim=-1)
    r, x, y, z = q.unbind(-1)
    R = torch.stack([torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y)], -1),
                     torch.stack([2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x)], -1),
                     torch.stack([2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], -1)], -2)
    c2w = torch.eye(4, dtype=torch.float64).repeat(C, 1, 1)
    c2w[:, :3, :3], c2w[:, :3, 3] = R, torch.randn(C, 3, generator=g, dtype=torch.float64)
    return torch.linalg.inv(c2w).transpose(1, 2).float().contiguous().cuda()


def bench_camera_step(C, reps=500):
    scene = synthetic.to_device(synthetic.make_scene(1000, 64, 96, 4, seed=0), "cuda")
    step = SplatTrainStep(scene, 64, 96, sh_degree=3, w_pearson=0.0)
    step.enable_camera_learning(random_viewmats(C, C), CameraLRs(1e-4, 1e-4))
    step.view_grad.normal_()
    it = [0]

    def one():
        step.collect_camera_grad(it[0] % C)
        step.camera_step(it[0])
        it[0] += 1

    for _ in range(20):
        one()
    t_step = timed_ms(one, reps)
    lib, cam, s = _lib.load(), step.cameras, _lib.stream_ptr()
    idx = torch.zeros(1, dtype=torch.int32, device="cuda")

    def kernels():
        _lib.check(lib.rdg_camera_grad(1, _lib.ptr(idx), _lib.ptr(cam["slots"]), _lib.ptr(cam["param"]), C, _lib.ptr(cam["grad"]),
                                       _lib.ptr(cam["error"]), s))
        _lib.check(lib.rdg_camera_adam(_lib.ptr(cam["param"]), _lib.ptr(cam["grad"]), _lib.ptr(cam["exp_avg"]),
                                       _lib.ptr(cam["exp_avg_sq"]), C, 1000, 1e-4, 1e-4, 0.9, 0.999, 1e-15, 1.0,
                                       _lib.ptr(cam["viewmats"]), s))

    for _ in range(20):
        kernels()
    return {"C": C, "camera_step_ms": round(t_step, 5), "kernels_ms": round(timed_ms(kernels, 5 * reps), 5)}


def bench_config4(rounds=6, steps=20):
    n, H, W, T, V = synthetic.CONFIGS["c4_iphone"]
    scene = synthetic.to_device(synthetic.make_scene(n, H, W, T, seed=0), "cuda")
    step = SplatTrainStep(scene, H, W, sh_degree=3, w_pearson=0.05)
    cams = [synthetic.make_camera(v, V, H, W, T) for v in range(V)]
    vms = torch.stack([c.world_view_transform.t().contiguous() for c in cams]).cuda()
    pms = [c.projection_matrix.t().contiguous().cuda() for c in cams]
    bts = [step.p("table")[c.time_index].contiguous() for c in cams]
    g = torch.Generator(device="cuda").manual_seed(1)
    gts = [torch.rand(3, H, W, device="cuda", generator=g) for _ in range(V)]
    gtd = [torch.rand(1, H, W, device="cuda", generator=g) + 1.0 for _ in range(V)]
    step.enable_camera_learning(vms, CameraLRs(1e-5, 1e-5))   # small rates: the rendered views stay those of the plain arm
    k = [0]

    def plain():
        v = k[0] % V
        step.forward_backward(vms[v], pms[v], cams[v].tanfovx, cams[v].tanfovy, bts[v], gts[v], gtd[v])
        k[0] += 1

    def learned():
        v = k[0] % V
        step.forward_backward(None, pms[v], cams[v].tanfovx, cams[v].tanfovy, bts[v], gts[v], gtd[v], camera=v)
        step.camera_step(k[0])
        k[0] += 1

    for fn in (plain, learned):
        for _ in range(5):
            fn()
    res = {"plain": [], "camera": []}
    for _ in range(rounds):
        res["plain"].append(timed_ms(plain, steps))
        res["camera"].append(timed_ms(learned, steps))
    med = {key: statistics.median(v) for key, v in res.items()}
    return {"config": "c4_iphone", "steps_per_run": steps, "runs": rounds, "plain_ms_median": round(med["plain"], 4),
            "camera_ms_median": round(med["camera"], 4), "delta_ms": round(med["camera"] - med["plain"], 4),
            "plain_ms_runs": [round(x, 4) for x in res["plain"]], "camera_ms_runs": [round(x, 4) for x in res["camera"]]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("camera_bench.py needs a CUDA device")
    name, power = gpu_identity()
    out = {"device": name, "power_limit": power, "camera_step": [bench_camera_step(C) for C in (100, 2000)],
           "step": bench_config4()}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
