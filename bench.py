#!/usr/bin/env python
"""bench.py - train iterations/sec of the dynamic-splatting hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c4_iphone] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one camera-time view per GPU:
deformation + preprocess + binning + blend forward + (L1 + D-SSIM + Pearson depth + alpha
term) + full backward to every Gaussian parameter, the motion coefficients, B(t) and the
motion table (+ the NCCL allreduce of the flat gradient buffer when N > 1).  The optimiser
is not part of BASELINE.json's metric ("raster fwd+bwd+loss"); `--adam` adds the fused Adam.

`value`  : whole-job iterations/s with that step's inputs (camera, targets) resident in HBM.
`e2e`    : same metric with the step's inputs (view + projection matrices, B(t), target image
           and depth) copied from pinned host memory and the loss read back inside the
           timed region.
`roofline`: the dominant kernel (largest share of the step, timed with CUDA events on the
           launching stream inside the timed region) against MEASURED_PEAKS.json.
`e2e_dropin`: the same step through the ZERO-CHANGE integration a RoDyGS user gets by pointing `diff_gauss_pose` at this
           repo: activated + concatenated tensors -> GaussianRasterizer (autograd Function, per-call allocation, the host
           read of num_rendered) -> rodygs_b200.losses -> loss.backward(), host-fed like `e2e`.
`cpu_baseline` / `--impl reference`: the PyTorch-CPU oracle (oracle/) on a bounded sample of the workload - a 256x256
           window at the workload's Gaussian density per tile - extrapolated to the full workload by algorithmic bytes
           (`"extrapolated": true`; `steps` / `warmup` are the frames actually run).
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last timed step returned to its caller as DIR/<name>.npy
           (see dump_outputs), so that two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

UNIT = "it/s"


def metric_name(cfg: str, forward_only: bool = False) -> str:
    """BASELINE.json's metric string for its quoted configuration (c4); the other configs name their own shape."""
    from rodygs_b200 import synthetic
    N, H, W, T, _ = synthetic.CONFIGS[cfg]
    shape = "1080p" if (H, W) == (1080, 1920) else f"{W}x{H}"
    n = f"{N / 1e6:g}M" if N >= 1_000_000 else f"{N // 1000}K"
    if forward_only:
        return f"forward-only render frames/sec at {shape}/{n} Gaussians; % HBM roofline"
    return f"train iters/sec (raster fwd+bwd+loss) at {shape}/{n} Gaussians; % HBM roofline"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            with open(path) as f:
                return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons, sampled every 20 ms from before the warm-up; stop(t0, t1) reports the samples
    that arrived DURING the timed region [t0, t1] (time.time() stamps)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "20"], stdout=subprocess.PIPE, text=True, bufsize=1)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float = 0.0, t1: float = float("inf")):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def parse(lines):
            sm, mx, reasons = [], [], set()
            for _, ln in lines:
                parts = [p.strip() for p in ln.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    sm.append(float(parts[1]))
                    mx.append(float(parts[2]))
                except ValueError:
                    continue
                for name, val in zip(names, parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons
        inside = [ln for ln in self.lines if t0 - 0.02 <= ln[0] <= t1 + 0.03]
        sm, mx, reasons = parse(inside)
        where = "timed region"
        if not sm:                       # a region shorter than the sampling period: fall back to the whole run (warm-up included)
            sm, mx, reasons = parse(self.lines)
            where = "whole run (no sample fell inside the timed region)"
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "period_ms": 20, "window": where}


# ------------------------------------------------------------------------------------ CPU arm
def sample_shape(cfg: str):
    """The bounded CPU sample of workload `cfg`: a 256x256-pixel window (256 tiles) with the workload's own number of
    Gaussians per tile (N' = N * 256 / tiles - the scene generator draws scales for a fixed screen radius, so the per-tile
    list length, which is what the blend cost depends on, matches: 736 entries per tile against 723 at BASELINE config 4),
    same T, same SH degree, same loss terms.  BASELINE config 1 (10K Gaussians, 256x256, CPU-sized) is its own sample."""
    from rodygs_b200 import synthetic
    Nf, Hf, Wf, T, _ = synthetic.CONFIGS[cfg]
    tiles_f = ((Hf + 15) // 16) * ((Wf + 15) // 16)
    if cfg == "c1_cpu":
        return Nf, Hf, Wf, T, tiles_f
    return max(1000, int(round(Nf * 256 / tiles_f))), 256, 256, T, tiles_f


def workload_counts(cfg: str, sh_degree: int = 3):
    """(N, visible V, dynamic N_d, duplicates D, pixels P) of the FULL workload's first view, counted on the CPU with the
    oracle's preprocess (radii > 0, sum of tiles_touched; bit-exact with the CUDA path by the parity contract) - what the
    sample's rate is extrapolated with, instead of assumed ratios."""
    from oracle import deform_oracle as do, splat_oracle as so
    from rodygs_b200 import synthetic
    N, H, W, T, _ = synthetic.CONFIGS[cfg]
    with torch.no_grad():
        sc = synthetic.make_scene(N, H, W, T, seed=0)
        cam = synthetic.make_camera(0, 8, H, W, T)
        st, dy = do.RawGaussians(**sc["static"]), do.RawGaussians(**sc["dynamic"])
        xyz, op, scl, rot, feat = do.assemble(st, dy, sc["motion_coeff"].squeeze(1), sc["table"][cam.time_index], sc["table"],
                                              sc["time_ind"].long(), 1.0, True)
        settings = so.Settings(H, W, cam.tanfovx, cam.tanfovy, torch.zeros(3), 1.0, cam.projection_matrix.t().contiguous(), 0)
        pp = so.preprocess(xyz, scl, rot, op, feat[:, :1].contiguous(), None, cam.world_view_transform.t().contiguous(), settings)
    return N, int((pp.radii > 0).sum()), N // 2, int(pp.tiles_touched.long().sum()), H * W


def cpu_oracle_rate(cfg: str = "c4_iphone", frames: int = 3, warmup: int = 1, sh_degree: int = 3, w_local: float = 0.15):
    """PyTorch-CPU oracle (fwd + full reference loss + bwd, all host threads) on `frames` frames of sample_shape(cfg).
    Returns (it/s at the sample, description, algorithmic bytes per iteration of the sample, per-frame seconds)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle import deform_oracle as do, loss_oracle as lo, splat_oracle as so
    from rodygs_b200 import synthetic
    torch.set_num_threads(os.cpu_count() or 1)
    N, H, W, T, tiles_f = sample_shape(cfg)
    sc = synthetic.make_scene(N, H, W, T, seed=0)
    g = torch.Generator().manual_seed(99)
    gt = torch.rand(3, H, W, generator=g)
    gt_d = torch.rand(1, H, W, generator=g)
    n_box = int(0.5 * (H // 128) * (W // 128))
    w_alpha = 0.01 if cfg == "c4_iphone" else 0.0
    times, stats = [], None
    for f in range(-warmup, frames):          # negative frames = warm-up
        cam = synthetic.make_camera(max(f, 0) % 8, 8, H, W, T)
        t0 = time.perf_counter()
        st = do.RawGaussians(**{k: x.clone().requires_grad_(True) for k, x in sc["static"].items()})
        dy = do.RawGaussians(**{k: x.clone().requires_grad_(True) for k, x in sc["dynamic"].items()})
        coeff = sc["motion_coeff"].clone().requires_grad_(True)
        table = sc["table"].clone().requires_grad_(True)
        xyz, op, scl, rot, feat = do.assemble(st, dy, coeff.squeeze(1), table[cam.time_index], table,
                                              sc["time_ind"].long(), 1.0, True)
        vm = cam.world_view_transform.t().contiguous().requires_grad_(True)
        settings = so.Settings(H, W, cam.tanfovx, cam.tanfovy, torch.zeros(3), 1.0,
                               cam.projection_matrix.t().contiguous(), sh_degree)
        out = so.rasterize(xyz, torch.zeros(N, 3, requires_grad=True), feat, None, op, scl, rot, vm, settings)
        loss = lo.photometric(out.color, gt) + 0.05 * lo.pearson_depth(out.depth, gt_d) + w_alpha * (1 - out.alpha).mean()
        if n_box > 0 and w_local:
            x0 = torch.randint(0, H - 128, (n_box,), generator=g)
            y0 = torch.randint(0, W - 128, (n_box,), generator=g)
            loss = loss + w_local * lo.local_pearson_depth(out.depth, gt_d, x0, y0, 128)
        loss.backward()
        dt = time.perf_counter() - t0
        if f >= 0:
            times.append(dt)
            stats = (N, int((out.radii > 0).sum()), N // 2, int(out.bn.keys.numel()), H * W)
    rate = len(times) / sum(times)
    K = (sh_degree + 1) ** 2
    nbytes = synthetic.algorithmic_bytes(*stats, sh_coeffs=K)
    desc = (f"oracle (PyTorch-CPU, fp32) on a {256 / tiles_f:.4f} sample of {cfg} at the same Gaussian density per tile: {N} "
            f"Gaussians (50% dynamic), {H}x{W} window ({(H // 16) * (W // 16)} of {tiles_f} tiles, {stats[3] / ((H // 16) * (W // 16)):.0f} "
            f"list entries per tile), T={T}, SH degree {sh_degree}, {len(times)} frames fwd+loss+bwd after {warmup} warm-up frame(s); "
            f"{rate:.3f} it/s at that size")
    return rate, desc, nbytes, times


def run_reference(args, rank):
    """The reference arm: the oracle port on the host cores.  One step = one frame of the bounded sample; the frames actually
    run are reported as `steps` / `warmup` (at most 24 + 2, so that the arm ends within a few minutes whatever K the driver
    asks for), and the rate is extrapolated to the full workload by algorithmic bytes with the workload's own counts."""
    if rank != 0:
        return
    from rodygs_b200 import synthetic
    frames, warm = max(1, min(args.steps, 24)), max(1, min(args.warmup, 2))
    rate, desc, sample_bytes, times = cpu_oracle_rate(args.config, frames, warm, args.sh_degree)
    counts = workload_counts(args.config, args.sh_degree)
    full_bytes = synthetic.algorithmic_bytes(*counts, sh_coeffs=(args.sh_degree + 1) ** 2)
    value = rate * sample_bytes / full_bytes
    cores = torch.get_num_threads()
    ts = sorted(times)
    line = {
        "impl": "reference", "metric": metric_name(args.config), "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": frames, "warmup": warm, "requested_steps": args.steps, "requested_warmup": args.warmup,
        "ms_per_step": 1000.0 / value, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "extrapolated": True,
        "config": {"workload": workload_name(args.config, args.sh_degree),
                   "note": "CPU arm: 256x256-pixel window at the workload's Gaussian density per tile; value = sample rate x "
                           "(sample algorithmic bytes / workload algorithmic bytes), the workload's V and D counted with the oracle's preprocess",
                   "workload_counts": dict(zip(("n", "visible", "dynamic", "duplicates", "pixels"), counts))},
        "sample": {"ms_per_frame_median": 1000.0 * ts[len(ts) // 2], "ms_per_frame_min": 1000.0 * ts[0], "ms_per_frame_max": 1000.0 * ts[-1],
                   "it_per_s": rate, "algorithmic_bytes": sample_bytes, "workload_algorithmic_bytes": full_bytes},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": desc + f"; scaled by algorithmic bytes {sample_bytes / full_bytes:.3e} to {args.config}",
                         "sample_value": rate},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_name(cfg, sh_degree=3):
    from rodygs_b200 import synthetic
    N, H, W, T, views = synthetic.CONFIGS[cfg]
    return f"{cfg}: {N} Gaussians (50% dynamic), {W}x{H}, T={T}, SH degree {sh_degree}, 1 camera-time view per GPU per step"


# ------------------------------------------------------------------------------------ GPU arm
DUMP_ROWS = 16384          # Gaussians per model in the seeded sample of the per-Gaussian outputs
DUMP_LIMIT = 64 << 20      # bytes written by --dump-outputs


def dump_outputs(step, out_dir: str, forward_only: bool, with_sh: bool) -> None:
    """What the last SplatTrainStep.forward_backward left for its caller, as float32 / float64 .npy files in out_dir.
    In full: the colour / depth / alpha maps and (training step) the loss parts, dL/dV, dL/dtable and dL/dB(t).  The full
    per-Gaussian gradients of the flagship workload are ~0.5 GB, so radii, dL/dmeans2D and every per-Gaussian parameter
    gradient are written at a fixed, seeded sample of DUMP_ROWS Gaussians per model (indices in index_<model>.npy).
    with_sh=False: dL/dSH was left in its factored form by the data-parallel exchange and is not written."""
    import numpy as np
    from rodygs_b200.trainer import PARAM_ORDER
    color, depth, alpha, radii = step.last_outputs
    out = {"color": color, "depth": depth, "alpha": alpha}
    if not forward_only:
        out.update(loss_parts=step.loss_parts, grad_viewmatrix=step.view_grad, grad_table=step.g("table"),
                   grad_basis_t=step.g("basis_t"))
    for tag, n, first in (("static", step.ns, 0), ("dynamic", step.nd, step.ns)):
        if n == 0:
            continue
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
        out[f"index_{tag}"] = idx.double()
        rows = idx.to(radii.device)
        out[f"radii_{tag}"] = radii[first + rows]
        if forward_only:
            continue
        out[f"grad_means2D_{tag}"] = step.means2D_grad[first + rows]
        names = [k for k in PARAM_ORDER if with_sh or not k.startswith("features")]
        for k in names + (["motion_coeff"] if tag == "dynamic" else []):
            out[f"grad_{tag}_{k}"] = step.g(k if k == "motion_coeff" else f"{tag}.{k}")[rows]
    arrays = {k: v.detach().cpu().numpy().astype(np.float64 if v.dtype == torch.float64 else np.float32) for k, v in out.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"bench.py: --dump-outputs would write {total / 2**20:.1f} MB (limit {DUMP_LIMIT >> 20} MB)")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from rodygs_b200 import _lib, engine, synthetic
    from rodygs_b200.trainer import SplatTrainStep

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    # the step draws its local-Pearson boxes on the device; torch seeds CUDA generators differently in every process, so
    # seed it to give every run with the same arguments the same inputs
    torch.cuda.manual_seed(rank)
    lib = _lib.load()
    engine.config.sync_free = False   # target generation below sizes the duplicate buffers exactly
    N, H, W, T, _ = synthetic.CONFIGS[args.config]
    if args.n_gaussians:
        N = args.n_gaussians
    scene_cpu = synthetic.make_scene(N, H, W, T, seed=0)
    scene = synthetic.to_device(scene_cpu, dev)
    w_alpha = 0.01 if args.config in ("c4_iphone",) else 0.0
    step = SplatTrainStep(scene, H, W, sh_degree=args.sh_degree, w_pearson=0.05, w_alpha=w_alpha, device=dev,
                          w_local=0.0 if args.no_local_pearson else 0.15)
    n_views = max(8, world)
    my_views = [v for v in range(n_views) if v % world == rank] or [rank % n_views]
    cams = [synthetic.make_camera(v, n_views, H, W, T) for v in my_views]

    def cam_tensors(cam, device, pin=False):
        vm = cam.world_view_transform.t().contiguous()
        pm = cam.projection_matrix.t().contiguous()
        if pin:
            return vm.pin_memory(), pm.pin_memory()
        return vm.to(device), pm.to(device)

    # targets: render of a perturbed copy of the scene (SURVEY.md §8d), depth min-max normalised
    targets = []
    view_counts = []                  # (visible, duplicates) of every view this rank renders
    with torch.no_grad():
        pert = 0.01 * torch.randn(step.p("static.xyz").shape, generator=torch.Generator().manual_seed(1000)).to(dev)
        step.p("static.xyz").add_(pert)
        for cam in cams:
            vm, pm = cam_tensors(cam, dev)
            step.forward_backward(vm, pm, cam.tanfovx, cam.tanfovy, step.p("table")[cam.time_index].contiguous(),
                                  None, None, forward_only=True)
            color, depth, alpha, radii_v = step.last_outputs
            view_counts.append((int((radii_v > 0).sum().item()), int(step.last_state.num_rendered[0].item())))
            d = depth.clone()
            d = (d - d.min()) / (d.max() - d.min() + 1e-12)
            targets.append((color.clone(), d))
        step.p("static.xyz").sub_(pert)
    torch.cuda.synchronize()
    engine.config.sync_free = True    # the timed steps never synchronise the host

    dev_inputs = []
    host_inputs = []
    for cam, (gt, gtd) in zip(cams, targets):
        vm, pm = cam_tensors(cam, dev)
        bt = step.p("table")[cam.time_index].clone()
        dev_inputs.append((vm, pm, bt, gt, gtd, cam))
        hvm, hpm = cam_tensors(cam, None, pin=True)
        host_inputs.append((hvm, hpm, bt.cpu().pin_memory(), gt.cpu().pin_memory(), gtd.cpu().pin_memory(), cam))
    # staging buffers for the e2e leg
    st_vm, st_pm = torch.empty(4, 4, device=dev), torch.empty(4, 4, device=dev)
    st_bt = torch.empty_like(dev_inputs[0][2])
    st_gt, st_gtd = torch.empty_like(targets[0][0]), torch.empty_like(targets[0][1])
    host_loss = torch.empty(8, dtype=torch.float32).pin_memory()
    h2d_bytes = sum(t.numel() * 4 for t in (st_vm, st_pm, st_bt, st_gt, st_gtd))
    d2h_bytes = host_loss.numel() * 4

    # data-parallel exchange (world > 1): the ranks all-gather the 12-byte factors of dL/dSH and all-reduce the rest;
    # every rank needs the view matrix and B(t) of every rank's view of the step (rank-major order)
    factored = world > 1 and not args.plain_allreduce and not args.forward_only
    if args.bwd_parts < 0:
        # measured (profiles/README.md): pipelining the exchange pays on 2 GPUs (2.76 vs 2.86 ms/step) and on 4 (2.80 vs 2.87), not on 8
        # (3.03-3.10 vs 2.94-2.98: the NVLink ingress is busy for the whole tail either way)
        args.bwd_parts, args.bwd_order, args.bwd_parts_static = (4, "dst", 1) if world <= 4 else (0, args.bwd_order, args.bwd_parts_static)
    all_vm, all_bt = [], []
    if factored:
        step.enable_factored_exchange(views_per_rank=1, world_size=world, copy_engine_gather=not args.nccl_gather,
                                      bucketed=not args.no_bucketed, sm_reserve=args.sm_reserve, multicast=args.multicast,
                                      sm_partition=not args.no_sm_partition, allreduce=args.allreduce, allreduce_ctas=args.allreduce_ctas,
                                      bwd_parts=args.bwd_parts, bwd_order=args.bwd_order,
                                      bwd_parts_static=args.bwd_parts_static)
        for j in range(len(my_views)):
            cs = [synthetic.make_camera(r + j * world, n_views, H, W, T) for r in range(world)]
            all_vm.append(torch.stack([c.world_view_transform.t().contiguous() for c in cs]).to(dev).contiguous())
            all_bt.append(torch.stack([step.p("table")[c.time_index] for c in cs]).contiguous())

    # N > 1: dL/dSH stays in its factored form and is consumed by the SH groups' Adam update (rdg_sh_adam_views); the timed step
    # ends when every rank holds the gathered factors and the all-reduced remaining range, i.e. everything its optimiser needs
    defer_sh = factored and not args.materialize_sh
    with_opt = [False]
    adam_state = None
    if args.adam:
        adam_state = (torch.zeros_like(step.params), torch.zeros_like(step.params))
    it_count = [0]

    # e2e input pipeline: two staging slots filled from pinned host memory on a copy stream, one step
    # ahead of the compute stream (the H2D copies are inside the timed region, overlapped with compute)
    copy_stream = torch.cuda.Stream()
    slots = [(st_vm, st_pm, st_bt, st_gt, st_gtd),
             tuple(torch.empty_like(t) for t in (st_vm, st_pm, st_bt, st_gt, st_gtd))]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def prefetch(k):
        src = host_inputs[k % len(host_inputs)][:5]
        s = k % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s])
            for dst, h in zip(slots[s], src):
                dst.copy_(h, non_blocking=True)
            ready[s].record(copy_stream)

    cur_stream = torch.cuda.current_stream()   # looked up once: torch.cuda.current_stream() costs ~15 us per call

    graphs = [None, None]     # e2e leg, one GPU: the step captured as a CUDA graph per staging slot (see after the main leg)

    def one_step(k, e2e=False):
        vm, pm, bt, gt, gtd, cam = (host_inputs if e2e else dev_inputs)[k % len(dev_inputs)]
        if e2e:
            if k == 0:
                prefetch(0)
            cur_stream.wait_event(ready[k % 2])
            vm, pm, bt, gt, gtd = slots[k % 2]
        if e2e and graphs[k % 2] is not None:
            graphs[k % 2].replay()
        else:
            step.forward_backward(vm, pm, cam.tanfovx, cam.tanfovy, bt, gt, gtd, forward_only=args.forward_only,
                                  dcolor_slot=0 if factored else None)
        if e2e:
            consumed[k % 2].record(cur_stream)
            prefetch(k + 1)    # enqueued after this step's launches: the GPU is never idle while the copies are set up
        if world > 1 and not args.forward_only:   # config 5 (inference): replicas only, no collective
            if args.plain_allreduce:
                step.allreduce_grads(1.0 / world)
            else:
                j = k % len(dev_inputs)
                step.exchange_grads(all_vm[j], all_bt[j], defer_sh=defer_sh)
        if with_opt[0]:
            it_count[0] += 1
            step.optimizer_step("static", it_count[0])
            step.optimizer_step("dynamic", it_count[0])
        if adam_state is not None:
            it_count[0] += 1
            _lib.check(lib.rdg_adam(step.params.data_ptr(), step.grads.data_ptr(), adam_state[0].data_ptr(),
                                    adam_state[1].data_ptr(), step.params.numel(), 1.6e-4, 0.9, 0.999, 1e-15,
                                    it_count[0], 1.0, _lib.stream_ptr()))
        if e2e:
            host_loss.copy_(step.loss_parts, non_blocking=True)
            cur_stream.synchronize()   # the user reads the loss every step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n_steps, e2e=False, fn=None):
        """n_steps steps between barriers; returns (total ms = max over ranks, per-step ms of this rank from one CUDA event
        per step on the launching stream, wall-clock start / end of the region)."""
        fn = fn or one_step
        barrier()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_steps + 1)]
        t0 = time.time()
        evs[0].record()
        for k in range(n_steps):
            fn(k, e2e)
            evs[k + 1].record()
        barrier()
        t1 = time.time()
        ms = evs[0].elapsed_time(evs[-1])
        per_step = [evs[k].elapsed_time(evs[k + 1]) for k in range(n_steps)]
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, per_step, t0, t1

    def pct(xs):
        ys = sorted(xs)
        q = lambda f: ys[min(len(ys) - 1, int(f * len(ys)))]
        return {"median": q(0.5), "p10": q(0.1), "p90": q(0.9), "min": ys[0], "max": ys[-1], "n": len(ys)}

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()                     # before the warm-up: the 20 ms sampler is up and running when the timed region starts
    n_warm = max(args.warmup, 3)
    for k in range(n_warm):
        one_step(k)
    torch.cuda.synchronize()

    launches0 = int(lib.rdg_launch_count())
    step.enable_stage_timing()
    ms_total, per_step, t_region0, t_region1 = timed(args.steps)
    launches = int(lib.rdg_launch_count()) - launches0
    events = step.stage_events
    step.stage_events = None
    clocks = sampler.stop(t_region0, t_region1) if sampler else None
    if args.dump_outputs and rank == 0:    # before the other legs overwrite the step's buffers
        dump_outputs(step, args.dump_outputs, args.forward_only, with_sh=not defer_sh)

    # e2e leg (host buffers -> H2D -> step -> D2H loss).  One GPU: the step is replayed as a CUDA graph (one per staging
    # slot), so the GPU does not wait for Python to enqueue ~25 launches after every loss read.
    e2e_api = "rodygs_b200.trainer.SplatTrainStep.forward_backward (fused flat-buffer path)"
    same_fov = all(abs(c.tanfovx - cams[0].tanfovx) < 1e-12 and abs(c.tanfovy - cams[0].tanfovy) < 1e-12 for c in cams)
    if world == 1 and not args.forward_only and not args.adam and not args.no_graph and same_fov:
        try:
            for s_ in range(2):
                for dst, h in zip(slots[s_], host_inputs[s_ % len(host_inputs)][:5]):
                    dst.copy_(h)
                vm_, pm_, bt_, gt_, gtd_ = slots[s_]
                graphs[s_] = step.capture_forward_backward(vm_, pm_, cams[0].tanfovx, cams[0].tanfovy, bt_, gt_, gtd_)
            e2e_api = "rodygs_b200.trainer.SplatTrainStep.capture_forward_backward + CapturedStep.replay (the fused step as one CUDA graph)"
        except Exception as e:   # noqa: BLE001 - the eager step is the fallback
            print(f"bench: CUDA-graph capture of the step failed ({type(e).__name__}: {e}); e2e runs eagerly", file=sys.stderr)
            graphs[0] = graphs[1] = None
    for k in range(2):
        one_step(k, e2e=True)
    ms_e2e, per_step_e2e, _, _ = timed(args.steps, e2e=True)

    # ---- e2e through the drop-in API (zero-change integration): activated tensors -> GaussianRasterizer -> losses -> backward
    dropin = None
    if not args.forward_only and not args.no_dropin and world == 1:
        dropin = run_dropin_leg(args, step, host_inputs, cams, dev, timed, pct)

    # ---- optional per-stream kernel timeline of one step (torch.profiler / CUPTI; never inside the timed region) ----
    if args.timeline:
        from torch.profiler import profile, ProfilerActivity
        barrier()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for k in range(3):
                one_step(k)
            torch.cuda.synchronize()
        if rank == 0:
            evs = sorted([e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA], key=lambda e: e.time_range.start)
            starts = [e for e in evs if "preprocess_fwd" in e.name]
            lo = starts[-1].time_range.start if starts else evs[0].time_range.start
            with open(args.timeline, "w") as f:
                f.write(f"# one data-parallel step on rank 0 of {world} (torch.profiler): start us, duration us, kernel\n")
                for e in evs:
                    if e.time_range.start >= lo:
                        f.write(f"{e.time_range.start - lo:9.1f} {e.time_range.end - e.time_range.start:8.1f}  {e.name[:90]}\n")
        barrier()

    # ---- the motion-basis MLP (row a1), timed on its own: the scene's table is a stand-in for its output
    # (SURVEY.md §8d), so the network runs beside the step, not inside it ----
    mlp_info = None
    if not args.forward_only:
        from rodygs_b200 import deform
        mlp = step.attach_basis_mlp(deform.BasisMLP(128, 16, 26, False, device=dev), torch.arange(T, dtype=torch.float32) / T)
        keep_table, keep_bt = step.p("table").clone(), step.p("basis_t").clone()
        l0 = int(lib.rdg_launch_count())
        for _ in range(3):
            step.basis_forward(0.37)
            step.basis_backward()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        for k in range(args.steps):
            step.basis_forward(0.01 * k)
            step.basis_backward()
        ev1.record()
        torch.cuda.synchronize()
        mlp_info = {"ms_fwd_bwd": ev0.elapsed_time(ev1) / args.steps, "rows": T + 1, "params": mlp.n_params,
                    "launches_per_step": (int(lib.rdg_launch_count()) - l0) // (args.steps + 3),
                    "note": "rdg_basis_mlp_fwd + _bwd for B(t) and the T-row table; not part of ms_per_step"}
        step.p("table").copy_(keep_table)
        step.p("basis_t").copy_(keep_bt)

    # ---- the step INCLUDING the optimiser (GaussianAdam with the reference's groups, both models): not the metric, but it shows
    # what the factored dL/dSH costs / saves end to end (N > 1: the SH groups step straight from the gathered factors) ----
    opt_info = None
    if not args.forward_only and not args.adam:
        from rodygs_b200.optim import GaussianLRs
        keep = step.params.clone()
        step.attach_optimizer("static", GaussianLRs())
        step.attach_optimizer("dynamic", GaussianLRs(scaling_lr=0.001, motion_coeff_lr=1.6e-4))
        with_opt[0] = True
        n_opt = max(5, min(args.steps, 30))
        for k in range(3):
            one_step(k)
        ms_opt, per_step_opt, _, _ = timed(n_opt)
        with_opt[0] = False
        step.params.copy_(keep)
        del keep
        opt_info = {"ms_per_step": ms_opt / n_opt, "value": world * 1000.0 * n_opt / ms_opt, "unit": UNIT, "steps": n_opt,
                    "ms_per_step_stats": pct(per_step_opt),
                    "note": "fwd + loss + bwd" + (" + exchange" if world > 1 else "") + " + Adam over every parameter group of both models ("
                            + ("f_dc / f_rest from the gathered dL/dSH factors by rdg_sh_adam_views, the rest by rdg_adam_groups" if defer_sh
                               else "rdg_adam_groups") + "); not the headline metric"}

    # ---- per-stage device times from the events recorded inside the timed region ----
    stage_ms = {}
    prev = None
    for name, ev in events:
        if name != "start" and prev is not None:
            stage_ms[name] = stage_ms.get(name, 0.0) + prev.elapsed_time(ev)
        prev = ev
    stage_ms = {k: v / args.steps for k, v in stage_ms.items()}

    # algorithmic bytes use the MEAN visible / duplicate counts over the views this rank cycles through
    V = int(round(sum(c[0] for c in view_counts) / len(view_counts)))
    D = int(round(sum(c[1] for c in view_counts) / len(view_counts)))
    P = H * W
    nd = step.nd
    K = (args.sh_degree + 1) ** 2
    stage_bytes = {
        "preprocess_fwd": 52 * N + (41 + 12 * K) * V + 68 * nd,
        "bin": 8 * N + 20 * V + 44 * D,
        "blend_fwd": 44 * D + 28 * P,
        "loss": 48 * P + (12 * P if step.w[2] else 0),
        "blend_bwd": 44 * D + 44 * P + 48 * V,
        "preprocess_bwd": 100 * N + (48 + 24 * K) * V + 132 * nd,
    }
    total_bytes = synthetic.algorithmic_bytes(N, V, nd, D, P, K, forward_only=args.forward_only)
    peak, peak_src = load_peaks()
    dom = max((k for k in stage_ms if k in stage_bytes), key=stage_ms.get) if stage_ms else "blend_bwd"
    dom_ms = stage_ms.get(dom, float("nan"))
    achieved = stage_bytes[dom] / (dom_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(args.config, {}).get(dom)
        except Exception:
            traffic = None

    # FP32-issue view of the dominant kernel (the blend kernels are issue bound, not HBM bound): warp instructions per
    # launch from the committed ncu capture (deterministic for this workload) over the live kernel time, against
    # SMs x 4 schedulers x the SM clock sampled during the run
    issue = None
    try:
        winst = json.load(open(tpath)).get(args.config + "_warp_inst", {})
        prefixes = {"blend_bwd": ("blend_bwd_kernel",), "blend_fwd": ("blend_fwd_kernel",),
                    "preprocess_fwd": ("preprocess_fwd_kernel",), "preprocess_bwd": ("preprocess_bwd_kernel", "dtable2_kernel"),
                    "loss": ("ssim_fwd_kernel", "ssim_bwd_kernel")}.get(dom, ())
        n_inst = sum(v for k, v in winst.items() if k.startswith(prefixes)) if prefixes else 0
        if n_inst and N == synthetic.CONFIGS[args.config][0]:
            mhz = (clocks or {}).get("sm_mhz") or 1965.0
            peak_i = 148 * 4 * mhz * 1e6
            issue = {"bound": "fp32_issue", "warp_inst_per_launch": n_inst, "achieved": n_inst / (dom_ms * 1e-3) / 1e9,
                     "peak": peak_i / 1e9, "unit": "Gwarp-inst/s", "frac": n_inst / (dom_ms * 1e-3) / peak_i,
                     "source": "profiles/traffic.json (ncu smsp__inst_executed.sum)"}
    except Exception:
        issue = None

    if rank == 0:
        ms_step = ms_total / args.steps
        value = world * 1000.0 / ms_step
        e2e_value = world * 1000.0 / (ms_e2e / args.steps)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            rate, desc, sample_bytes, _ = cpu_oracle_rate(args.config, 3, 1, args.sh_degree, 0.0 if args.no_local_pearson else 0.15)
            scaled = rate * sample_bytes / total_bytes
            cpu = {"value": scaled, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                   "sample": desc + f"; scaled by algorithmic bytes ({sample_bytes / total_bytes:.3e}) to this workload",
                   "sample_value": rate}
        if factored:
            parallelism = (f"dp{world} (view-sharded; all-gather of the 12 B/Gaussian factors of dL/dSH + allreduce of the other gradients"
                           + ("" if args.no_bucketed else
                              (f" by the in-switch kernel rdg_allreduce_multimem, pipelined under the per-Gaussian backward ({len(step._bwd_plan)} launches, order {args.bwd_order}), "
                               f"{args.sm_reserve} SMs left to it" if step._ar_mode == "multimem" and step._bwd_plan is not None else
                               f" ({step._ar_mode}) per model under the other model's backward kernel, {args.sm_reserve} SMs left to the collective"))
                           + (", dL/dSH kept factored for the SH groups' fused Adam (rdg_sh_adam_views) - not materialised in the timed step)"
                              if defer_sh else ", dL/dSH rebuilt per rank)"))
        else:
            parallelism = f"dp{world} (view-sharded, allreduce of the flat gradient buffer)"
        line = {
            "metric": metric_name(args.config, args.forward_only),
            "value": value, "unit": UNIT if not args.forward_only else "frames/s", "n_gpus": world, "steps": args.steps, "warmup": n_warm,
            "ms_per_step": ms_step, "ms_per_step_stats": pct(per_step), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.config, args.sh_degree), "n_gaussians": N, "visible": V, "duplicates": D,
                       "sh_degree": args.sh_degree,
                       "loss": ("0.8 L1 + 0.2 D-SSIM + 0.05 global Pearson" + ("" if args.no_local_pearson else f" + 0.15 local Pearson ({step.n_local} boxes of 128x128)")
                                + (" + 0.01 mean(1 - alpha)" if w_alpha else "")) if not args.forward_only else "none (forward only)",
                       "pixels": P, "views_per_step": world, "l2": "inputs larger than L2 (params+SH 472 MB, sort buffers)",
                       "optimizer": "fused Adam in the timed region" if args.adam else "excluded (metric = raster fwd+bwd+loss)",
                       "sync_free": True, "parallelism": parallelism},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": ms_e2e / args.steps, "ms_per_step_stats": pct(per_step_e2e),
                    "api": e2e_api},
            "e2e_dropin": dropin,
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "kernel_ms": dom_ms, "algorithmic_bytes": stage_bytes[dom]},
            "issue_roofline": issue,
            "step_roofline": {"algorithmic_bytes": total_bytes, "achieved": total_bytes / (ms_step * 1e-3) / 1e9,
                              "frac": total_bytes / (ms_step * 1e-3) / 1e9 / peak,
                              "note": "whole step (all kernels + launch gaps) against the HBM peak"},
            "stage_ms": stage_ms,
            "basis_mlp": mlp_info,
            "with_optimizer": opt_info,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)


def run_dropin_leg(args, step, host_inputs, cams, dev, timed, pct):
    """One training step the way an UNMODIFIED RoDyGS trainer would run it on this library (SURVEY.md §8b): the activated,
    concatenated tensors of get_GS_properties (rodygs.py:68-113) -> GaussianRasterizationSettings / GaussianRasterizer
    (renderer.py:50-101; torch.autograd.Function, per-call allocation, the host read of num_rendered) -> the reference's loss
    functions from rodygs_b200.losses -> loss.backward().  Host-fed like `e2e`: the view's matrices and targets come from
    pinned host memory every step and the loss is read back."""
    from rodygs_b200 import engine, losses
    from rodygs_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    was = engine.config.sync_free
    engine.config.sync_free = False          # the drop-in API keeps the reference's one host read per forward
    try:
        with torch.no_grad():                # activated + concatenated leaves (static first, dynamic second, no deformation)
            cat = lambda k: torch.cat([step.p(f"static.{k}"), step.p(f"dynamic.{k}")], 0)
            xyz = cat("xyz").clone().requires_grad_(True)
            opac = torch.sigmoid(cat("opacity")).requires_grad_(True)
            scal = torch.exp(cat("scaling")).requires_grad_(True)
            rot = torch.nn.functional.normalize(cat("rotation")).requires_grad_(True)
            feat = torch.cat([cat("features_dc"), cat("features_rest")], 1).contiguous().requires_grad_(True)
        leaves = [xyz, opac, scal, rot, feat]
        n = xyz.shape[0]
        bg = torch.zeros(3, device=dev)
        slots = [tuple(torch.empty_like(t, device=dev) for t in host_inputs[0][:5]) for _ in range(2)]
        host_loss = torch.empty((), dtype=torch.float32).pin_memory()
        H, W = step.H, step.W
        n_box = step.n_local

        def one(k, e2e=True):
            hvm, hpm, hbt, hgt, hgtd, cam = host_inputs[k % len(host_inputs)]
            vm, pm, _, gt, gtd = slots[k % 2]
            vm.copy_(hvm, non_blocking=True); pm.copy_(hpm, non_blocking=True)
            gt.copy_(hgt, non_blocking=True); gtd.copy_(hgtd, non_blocking=True)
            for t in leaves:
                t.grad = None
            vm_leaf = vm.clone().requires_grad_(True)
            means2D = torch.zeros(n, 3, device=dev, requires_grad=True)
            st = GaussianRasterizationSettings(H, W, cam.tanfovx, cam.tanfovy, bg, 1.0, pm, args.sh_degree, False, False, True, True)
            color, depth, normal, alpha, radii, extra = GaussianRasterizer(st)(
                means3D=xyz, means2D=means2D, shs=feat, colors_precomp=None, opacities=opac, scales=scal, rotations=rot,
                cov3Ds_precomp=None, viewmatrix=vm_leaf)
            loss = losses.photometric_loss(color, gt, 0.8, 0.2) + 0.05 * losses.pearson_depth_loss(depth, gtd)
            if n_box > 0:
                loss = loss + 0.15 * losses.local_pearson_depth_loss(depth, gtd, 128, 0.5)
            loss.backward()
            host_loss.copy_(loss.detach(), non_blocking=True)
            torch.cuda.current_stream().synchronize()

        steps = max(5, min(args.steps, 30))
        for k in range(3):
            one(k)
        ms, per_step, _, _ = timed(steps, True, one)
        h2d = sum(t.numel() * 4 for t in (slots[0][0], slots[0][1], slots[0][3], slots[0][4]))
        return {"value": 1000.0 * steps / ms, "unit": UNIT, "ms_per_step": ms / steps, "ms_per_step_stats": pct(per_step), "steps": steps,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 + 8,
                "api": "diff_gauss_pose.GaussianRasterizer (drop-in) + rodygs_b200.losses + autograd; activated, concatenated "
                       "inputs, no fused deformation, dL/dSH written in full"}
    finally:
        engine.config.sync_free = was
        for t in (xyz, opac, scal, rot, feat):
            t.grad = None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--sh-degree", type=int, default=3, choices=[0, 1, 2, 3],
                    help="active SH degree (the reference trains at degree 0 for 15000 of 20000 iterations)")
    ap.add_argument("--no-local-pearson", action="store_true", help="leave the 0.15-weighted LocalPearsonDepthLoss out of the step (A/B)")
    ap.add_argument("--no-graph", action="store_true", help="e2e leg: enqueue the step eagerly instead of replaying its CUDA graph (A/B)")
    ap.add_argument("--no-dropin", action="store_true", help="skip the e2e_dropin leg (GaussianRasterizer + autograd)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c4_iphone")
    ap.add_argument("--n-gaussians", type=int, default=0)
    ap.add_argument("--adam", action="store_true")
    ap.add_argument("--forward-only", action="store_true", help="BASELINE config 5: inference render sweep")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--nccl-gather", action="store_true",
                    help="N>1: gather the dL/dSH factors with NCCL instead of copy-engine pulls over symmetric memory (A/B)")
    ap.add_argument("--no-bucketed", action="store_true",
                    help="N>1: one all-reduce of the non-SH range after the whole backward instead of one per model under the other model's kernel (A/B)")
    ap.add_argument("--multicast", action="store_true",
                    help="N>1: gather the dL/dSH factors with NVLS multicast stores from the producing kernel instead of copy-engine pushes (A/B; measured slower)")
    ap.add_argument("--sm-reserve", type=int, default=16,
                    help="N>1: SMs the persistent backward kernels leave to NCCL while the bucketed all-reduce runs beside them")
    ap.add_argument("--timeline", default="", help="write the kernel timeline of one step (rank 0, torch.profiler) to this file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the last step's outputs as DIR/<name>.npy (at most 64 MB; see dump_outputs)")
    ap.add_argument("--no-sm-partition", action="store_true",
                    help="N>1: size the persistent backward grids for 148 - sm_reserve SMs instead of the SM-partitioned chunk queue (A/B)")
    ap.add_argument("--bwd-parts", type=int, default=-1,
                    help="N>1, --allreduce multimem: launches of the dynamic model's per-Gaussian backward (pipelined exchange); 0: one bucket per model; "
                         "-1 (default): the measured best - pipelined (4 dynamic launches, static, dL/dtable) on 2 / 4 GPUs, one bucket per model on 8")
    ap.add_argument("--allreduce", default="multimem", choices=["nccl", "multimem", "symm_op"],
                    help="N>1: all-reduce of the non-SH gradient range: NCCL, the in-switch kernel rdg_allreduce_multimem, or torch's symm_mem op")
    ap.add_argument("--allreduce-ctas", type=int, default=32)
    ap.add_argument("--bwd-parts-static", type=int, default=2)
    ap.add_argument("--bwd-order", default="sdt", help="N>1 pipelined exchange: order of the static launch (s), the dynamic launches (d) and the dL/dtable reduction (t)")
    ap.add_argument("--materialize-sh", action="store_true",
                    help="N>1: rebuild dL/dSH of all views in the timed step (rdg_sh_grad_views) instead of leaving the factors to the fused SH Adam")
    ap.add_argument("--plain-allreduce", action="store_true",
                    help="N>1: all-reduce the whole flat gradient buffer instead of the factored SH exchange (A/B)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                         "(use --impl reference for the CPU oracle arm)")
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
