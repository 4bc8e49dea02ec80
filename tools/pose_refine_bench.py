"""Time test-time pose refinement: the captured loop (rodygs_b200.pose.refine_poses, one CUDA graph per iteration) against
the reference-shaped loop (the drop-in GaussianRasterizer + V(q, T) in torch with autograd + L2 + torch.optim.Adam, what
RoDyGS's PoseOptimizer runs), on the static half of BASELINE configs 2 and 4, alternating the two loops, and print one JSON
line with the GPU's name and power limit.

    python tools/pose_refine_bench.py [--iters 200] [--repeats 3] [--lr 1e-3] [--out FILE]

Per config and repeat: refine_poses(iters) and the reference loop for the same iterations from the same start pose, each
timed on the host around a device synchronise (set-up included: the sizing read, the eager warm-up iteration and the
capture of the captured loop); then `iters` replays of the captured graph alone between CUDA events (steady state).
Also imported by tests/test_pose_refine.py for the reference loop and the float64 restatement of V(q, T)."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rodygs_b200 import GaussianRasterizationSettings, GaussianRasterizer, pose, synthetic  # noqa: E402

CONFIGS = ("c2_kubric", "c4_iphone")


def view_from_pose(q: torch.Tensor, T: torch.Tensor) -> torch.Tensor:
    """V(q, T) in glm storage (V^T), differentiable, in the dtype of q: R = rot(q / |q|), V = [[R^T, -R^T T], [0, 0, 0, 1]]."""
    r, x, y, z = (q / q.norm()).unbind()
    R = torch.stack([torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y)]),
                     torch.stack([2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x)]),
                     torch.stack([2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)])])
    top = torch.cat([R, torch.zeros(3, 1, dtype=q.dtype, device=q.device)], 1)
    bottom = torch.cat([-(T @ R), torch.ones(1, dtype=q.dtype, device=q.device)]).unsqueeze(0)
    return torch.cat([top, bottom], 0)


def reference_loop(static, H, W, sh_degree, bg, projmat, tanfovx, tanfovy, gt, pose0, lr, iters):
    """The reference-shaped loop: returns (q, T, losses [iters], (dL/dq, dL/dT) of the first iteration)."""
    q = pose0[:4].clone().requires_grad_(True)
    T = pose0[4:].clone().requires_grad_(True)
    opt = torch.optim.Adam([q, T], lr=lr)
    rast = GaussianRasterizer(GaussianRasterizationSettings(H, W, tanfovx, tanfovy, bg, 1.0, projmat, sh_degree, False, False,
                                                            True, True))
    act = dict(means3D=static["xyz"], shs=torch.cat([static["features_dc"], static["features_rest"]], 1).contiguous(),
               opacities=torch.sigmoid(static["opacity"]), scales=torch.exp(static["scaling"]),
               rotations=F.normalize(static["rotation"], dim=-1))
    means2D = torch.zeros_like(static["xyz"])
    losses, first = [], None
    for _ in range(iters):
        color = rast(means2D=means2D, viewmatrix=view_from_pose(q, T), **act)[0]
        loss = ((color - gt) ** 2).mean()
        opt.zero_grad(set_to_none=True)
        loss.backward()
        if first is None:
            first = (q.grad.clone(), T.grad.clone())
        opt.step()
        losses.append(loss.detach())
    return q.detach(), T.detach(), torch.stack(losses), first


def gpu_identity():
    idx = torch.cuda.current_device()
    try:
        q = subprocess.run(["nvidia-smi", f"--id={idx}", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (s.strip() for s in q.split(","))
    except Exception as e:   # noqa: BLE001 - the number is still reported, with what is known
        name, power = torch.cuda.get_device_name(idx), f"unknown ({type(e).__name__})"
    return name, power


def _setup(config):
    n, H, W, T, _ = synthetic.CONFIGS[config]
    scene = synthetic.to_device(synthetic.make_scene(n, H, W, T, seed=0), "cuda")
    static = scene["static"]
    cam = synthetic.make_camera(0, 8, H, W, T)
    vm_true = cam.world_view_transform.t().contiguous().cuda()
    pm = cam.projection_matrix.t().contiguous().cuda()
    bg = torch.zeros(3, device="cuda")
    p_true = pose.pose_from_viewmatrix(vm_true[None])[0]
    rast = GaussianRasterizer(GaussianRasterizationSettings(H, W, cam.tanfovx, cam.tanfovy, bg, 1.0, pm, 3, False, False,
                                                            True, True))
    gt = rast(means3D=static["xyz"], means2D=torch.zeros_like(static["xyz"]),
              shs=torch.cat([static["features_dc"], static["features_rest"]], 1).contiguous(),
              opacities=torch.sigmoid(static["opacity"]), scales=torch.exp(static["scaling"]),
              rotations=F.normalize(static["rotation"], dim=-1), viewmatrix=vm_true)[0].detach()
    start = p_true.clone()
    start[4:] += torch.tensor([0.05, -0.03, 0.04], device="cuda")          # camera centre moved, rotation kept
    vm0 = view_from_pose(start[:4].double(), start[4:].double()).float().contiguous()
    return dict(static=static, H=H, W=W, cam=cam, pm=pm, bg=bg, gt=gt, start=start, vm0=vm0, n_static=static["xyz"].shape[0])


def _wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def bench_config(config, iters, repeats, lr):
    s = _setup(config)
    cam = s["cam"]
    ours_ms, ref_ms, replay_ms = [], [], []
    ours = ref = None

    def run_ours():
        return pose.refine_poses(s["static"], s["H"], s["W"], 3, s["bg"], s["vm0"][None], s["pm"][None], cam.tanfovx, cam.tanfovy,
                                 s["gt"][None], lr, iters)

    def run_ref():
        return reference_loop(s["static"], s["H"], s["W"], 3, s["bg"], s["pm"], cam.tanfovx, cam.tanfovy, s["gt"], s["start"],
                              lr, iters)

    run_ours()           # warm-up of both paths (module loading, allocator)
    run_ref()
    for _ in range(repeats):
        t, ours = _wall(run_ours)
        ours_ms.append(t / iters)
        t, ref = _wall(run_ref)
        ref_ms.append(t / iters)
    # steady state of the captured loop: replays of the graph alone (after the last update the counter blocks further
    # updates, every replay still renders, differentiates and runs the guard)
    view = pose.ViewArgs(height=s["H"], width=s["W"], tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, scale_modifier=1.0, sh_degree=3,
                         viewmatrix=s["vm0"], projmatrix=s["pm"], bg=s["bg"])
    loop = pose._PoseLoop(pose._static_set(s["static"]), view, s["gt"], s["start"].contiguous(), lr, 1)
    loop.run()
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            loop.graph.replay()
        b.record()
        torch.cuda.synchronize()
        replay_ms.append(a.elapsed_time(b) / iters)
    q_diff = float((ours[0][0] - view_from_pose(ref[0].double(), ref[1].double()).float()).abs().max())
    med = lambda v: sorted(v)[len(v) // 2]   # noqa: E731
    return {"config": config, "n_static": s["n_static"], "height": s["H"], "width": s["W"], "iters": iters, "lr": lr,
            "captured_ms_per_iter": round(med(ours_ms), 4), "captured_ms_per_iter_all": [round(x, 4) for x in ours_ms],
            "graph_replay_ms_per_iter": round(med(replay_ms), 4),
            "reference_ms_per_iter": round(med(ref_ms), 4), "reference_ms_per_iter_all": [round(x, 4) for x in ref_ms],
            "speedup": round(med(ref_ms) / med(ours_ms), 2),
            "final_loss_captured": float(ours[1][0, -1]), "final_loss_reference": float(ref[2][-1]),
            "initial_loss": float(ours[1][0, 0]), "max_abs_diff_final_V": q_diff}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--lr", type=float, default=1e-3)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pose_refine_bench: needs a CUDA device (times are measured on the GPU only)")
    name, power = gpu_identity()
    rows = [bench_config(c, args.iters, args.repeats, args.lr) for c in args.configs.split(",")]
    line = {"tool": "pose_refine_bench", "gpu": name, "power_limit": power, "results": rows}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")
    if not all(math.isfinite(r["final_loss_captured"]) for r in rows):
        raise SystemExit("pose_refine_bench: the captured loop produced a non-finite loss")


if __name__ == "__main__":
    main()
