"""Tracking the BASELINE config-5 scene (6 M Gaussians, 50 % dynamic, 1920x1080, T = 100, SH degree 3) into 8 targets, with
CUDA events around work that ends in a device synchronise:

* track:  SplatTrainStep.track_maps of one source view into 8 target camera-times (one preprocess + binning of the source,
          then rdg_track_attrs + rdg_blend_fwd per target and one rdg_track_project);
* render: SplatTrainStep.render_views of 8 views, the yardstick for what a blend of this scene costs;
* staged: track_maps again with an event after each stage (engine.track's stage_hook), split per target into attrs / blend /
          project, plus the source stage per call.

The arms alternate run by run after a warm-up of each; the scene (about 1.8 GB of parameters) is far larger than the L2.

Prints one JSON line with the device name and power limit.  Usage: python tools/track_bench.py [--runs R] [--out file.json]"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rodygs_b200 import engine, synthetic  # noqa: E402
from rodygs_b200.trainer import SplatTrainStep  # noqa: E402
from camera_bench import gpu_identity  # noqa: E402
from render_bench import timed_ms  # noqa: E402

M = 8


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    N, H, W, T, _ = synthetic.CONFIGS["c5_infer"]
    scene = synthetic.to_device(synthetic.make_scene(N, H, W, T, seed=0), "cuda")
    step = SplatTrainStep(scene, H, W, sh_degree=3, w_pearson=0.0)
    del scene
    cams = [synthetic.make_camera(v, M, H, W, T) for v in range(M)]
    vms = torch.stack([c.world_view_transform.t().contiguous() for c in cams]).cuda()
    pms = torch.stack([c.projection_matrix.t().contiguous() for c in cams]).cuda()
    bts = torch.stack([step.p("table")[c.time_index] for c in cams]).contiguous()
    fx, fy = cams[0].tanfovx, cams[0].tanfovy
    src = (vms[0], pms[0], fx, fy, bts[0])

    def track():
        return step.track_maps(*src, vms, pms, bts)

    def render():
        return step.render_views(vms, pms, fx, fy, bts)

    marks = []

    def hook(name):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        marks.append((name, ev))

    def staged():
        marks.clear()
        hook("start")
        scene_, view = step._scene_view(vms[0], pms[0], fx, fy, None)
        engine.track(scene_, view, bts[0], vms, pms, bts, stage_hook=hook)

    arms = {"track": track, "render_views": render, "track_staged": staged}
    for fn in arms.values():          # warm-up of every shape the timed runs use
        for _ in range(2):
            fn()
    alpha = track()[2]
    covered = float((alpha > 0).float().mean())
    times = {k: [] for k in arms}
    stages = {"source": [], "attrs": [], "blend": [], "project": []}
    for _ in range(args.runs):
        for k, fn in arms.items():
            times[k].append(timed_ms(fn) / M)
            if k == "track_staged":
                per = {s: 0.0 for s in stages}
                for (_, a), (name, b) in zip(marks, marks[1:]):
                    per[name] += a.elapsed_time(b)
                stages["source"].append(per["source"])
                for s in ("attrs", "blend", "project"):
                    stages[s].append(per[s] / M)
    name, power = gpu_identity()
    med = statistics.median
    res = {"tool": "track_bench", "device": name, "power_limit": power, "workload": "c5_infer", "n": step.ns + step.nd,
           "height": H, "width": W, "num_times": T, "sh_degree": 3, "targets": M, "runs": args.runs,
           "source_alpha_covered": covered,
           "per_target_ms": {k: {"median": med(v), "min": min(v), "max": max(v)} for k, v in times.items()},
           "stage_ms": {"source_per_call": {"median": med(stages["source"]), "min": min(stages["source"])},
                        **{f"{s}_per_target": {"median": med(stages[s]), "min": min(stages[s]), "max": max(stages[s])}
                           for s in ("attrs", "blend", "project")}}}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
