"""Rendering 8 views of the BASELINE config-5 scene (6 M Gaussians, 50 % dynamic, 1920x1080, T = 100, SH degree 3), with
CUDA events around work that ends in a device synchronise:

* batched: SplatTrainStep.render_views of the 8 views (one rdg_preprocess_fwd_views, one host read, bin + blend per view);
* loop:    engine.render_forward of the same 8 views one by one (rdg_preprocess_fwd + its host read + bin + blend each);

and the preprocess stage of each arm alone (rdg_preprocess_fwd_views of the 8 views against 8 rdg_preprocess_fwd launches).
The arms alternate run by run after a warm-up of both; the scene (about 1.8 GB of parameters) is far larger than the L2.
The outputs of the two arms are compared bit for bit first.

Prints one JSON line with the device name and power limit.  Usage: python tools/render_bench.py [--runs R] [--out file.json]"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rodygs_b200 import _lib, engine, synthetic  # noqa: E402
from rodygs_b200.trainer import SplatTrainStep  # noqa: E402
from camera_bench import gpu_identity  # noqa: E402

V = 8


def timed_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    N, H, W, T, _ = synthetic.CONFIGS["c5_infer"]
    scene = synthetic.to_device(synthetic.make_scene(N, H, W, T, seed=0), "cuda")
    step = SplatTrainStep(scene, H, W, sh_degree=3, w_pearson=0.0)
    del scene
    cams = [synthetic.make_camera(v, V, H, W, T) for v in range(V)]
    vms = torch.stack([c.world_view_transform.t().contiguous() for c in cams]).cuda()
    pms = torch.stack([c.projection_matrix.t().contiguous() for c in cams]).cuda()
    bts = torch.stack([step.p("table")[c.time_index] for c in cams]).contiguous()
    fx, fy = [c.tanfovx for c in cams], [c.tanfovy for c in cams]
    pairs = [step._scene_view(vms[v], pms[v], fx[v], fy[v], bts[v]) for v in range(V)]

    def batched():
        return step.render_views(vms, pms, fx, fy, bts)

    def loop():
        return [engine.render_forward(sc, vw, keep_for_backward=False)[:4] for sc, vw in pairs]

    got, ref = batched(), loop()
    identical = all(torch.equal(got[k], torch.stack([r[k] for r in ref])) for k in range(4))
    del got, ref

    # the preprocess stage alone, into preallocated geometry buffers
    lib, stream, n = _lib.load(), _lib.stream_ptr(), step.ns + step.nd
    tiles = engine.tiles_of(H, W)
    geoms = [engine._alloc_geom(n, "cuda", tile_count=torch.empty(tiles + 1, dtype=torch.int32, device="cuda")) for _ in range(V)]
    gm = (_lib.RdgGeom * V)(*[engine._geom_struct(g) for g in geoms])
    vw = (_lib.RdgView * V)(*[engine._view_struct(p[1]) for p in pairs])
    sc_views = engine._scene_struct(step._scene_view(vms[0], pms[0], fx[0], fy[0], None)[0])
    sc_single = [engine._scene_struct(p[0]) for p in pairs]

    def pre_batched():
        _lib.check(lib.rdg_preprocess_fwd_views(C.byref(sc_views), bts.data_ptr(), V, vw, gm, stream))

    def pre_loop():
        for v in range(V):
            _lib.check(lib.rdg_preprocess_fwd(C.byref(sc_single[v]), C.byref(vw[v]), C.byref(gm[v]), stream))

    arms = {"render_batched": batched, "render_loop": loop, "preprocess_batched": pre_batched, "preprocess_loop": pre_loop}
    for fn in arms.values():          # warm-up of every shape the timed runs use
        for _ in range(2):
            fn()
    times = {k: [] for k in arms}
    for _ in range(args.runs):
        for k, fn in arms.items():
            times[k].append(timed_ms(fn) / V)
    name, power = gpu_identity()
    res = {"tool": "render_bench", "device": name, "power_limit": power, "workload": "c5_infer", "n": n, "height": H,
           "width": W, "num_times": T, "sh_degree": 3, "views": V, "runs": args.runs, "bit_identical": identical,
           "per_view_ms": {k: {"median": statistics.median(v), "min": min(v), "max": max(v)} for k, v in times.items()}}
    pv = res["per_view_ms"]
    res["speedup_render"] = pv["render_loop"]["median"] / pv["render_batched"]["median"]
    res["speedup_preprocess"] = pv["preprocess_loop"]["median"] / pv["preprocess_batched"]["median"]
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
