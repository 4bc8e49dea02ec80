"""Engine-level training step on flat parameter / gradient buffers: the per-iteration
hot loop of /root/reference/src/trainer/rodygs.py:198-310 (get_GS_properties -> render
-> MultiLoss -> loss.backward) as ONE explicit sequence of C-ABI calls - no autograd
graph, no concat, no host synchronisation, gradients written straight into one flat
fp32 buffer that the data-parallel allreduce consumes (SURVEY.md §8e).

Multi-GPU: one process per GPU, every rank holds a full replica of the Gaussians and
renders its own camera-time view(s); the only exchange step is the sum of the flat
gradient buffer (`torch.distributed.all_reduce`, NCCL over NVLink on the GPU box,
gloo in the CPU tests).  Pose gradients and the means2D sink stay rank-local.
"""
from __future__ import annotations

import ctypes as C
import copy
import math
import os
import sys
from typing import Dict, List, Optional, Tuple

import torch

from . import _lib, engine
from ._lib import check, ptr
from .engine import SceneArgs, SceneGrads, SetArgs, SetGrads, ViewArgs

PARAM_ORDER = ("xyz", "scaling", "rotation", "opacity", "features_dc", "features_rest")
# SplatTrainStep.state_dict(): the tag and version a loader checks before it reads anything else
CHECKPOINT_FORMAT, CHECKPOINT_VERSION = "rodygs_b200.SplatTrainStep", 1
STATS_FIELDS = ("grad_accum", "denom", "max_radii2D")


def flat_layout(n_static: int, n_dynamic: int, num_basis: int, num_times: int) -> Tuple[Dict[str, Tuple[int, Tuple[int, ...]]], int]:
    """name -> (float offset, shape) of every trainable tensor inside the flat buffer.
    Offsets are multiples of 64 floats (256 B) so that every slice is vector-aligned.  The SH blocks
    come last: everything before `sh_start(layout)` is what the data-parallel step all-reduces,
    the SH gradients are rebuilt from their 12-byte factors (see SplatTrainStep.exchange_grads)."""
    shapes = {}
    for tag, n in (("static", n_static), ("dynamic", n_dynamic)):
        shapes[f"{tag}.xyz"] = (n, 3)
        shapes[f"{tag}.scaling"] = (n, 3)
        shapes[f"{tag}.rotation"] = (n, 4)
        shapes[f"{tag}.opacity"] = (n, 1)
    shapes["motion_coeff"] = (n_dynamic, 1, num_basis)
    shapes["table"] = (num_times, num_basis, 7)
    shapes["basis_t"] = (num_basis, 7)
    sh_shapes = {}
    for tag, n in (("static", n_static), ("dynamic", n_dynamic)):
        sh_shapes[f"{tag}.features_dc"] = (n, 1, 3)
        sh_shapes[f"{tag}.features_rest"] = (n, 15, 3)
    layout, off = {}, 0
    for group in (shapes, sh_shapes):
        for name, shp in group.items():
            numel = 1
            for s in shp:
                numel *= s
            layout[name] = (off, shp)
            off += (numel + 63) // 64 * 64
    return layout, off


def sh_start(layout) -> int:
    """Float offset of the first SH block inside the flat buffer (= length of the all-reduced range)."""
    return layout["static.features_dc"][0]


def shard_views(n_views: int, world_size: int, rank: int) -> List[int]:
    """Round-robin split of a step's camera-time views over the ranks (SURVEY.md §8e)."""
    return [v for v in range(n_views) if v % world_size == rank]


# ReduceOp.AVG saves the scaling pass, but NCCL has no NVLS (in-switch) reduction for it (pre-multiplied sum) and falls back
# to a ring; RDG_AR_SUM=1 selects SUM + a scaling pass instead (A/B switch, see profiles/README.md)
AVG_ON_COLLECTIVE = os.environ.get("RDG_AR_SUM", "0") != "1"


def allreduce_flat(buf: torch.Tensor, scale: Optional[float] = None, group=None) -> torch.Tensor:
    """The data path's exchange step for a flat gradient range: in-place sum over the data-parallel group
    (NCCL on GPUs, gloo in the CPU tests), then an optional scale (1 / views for a mean over the step's
    views).  On NCCL a scale of exactly 1 / world_size rides on the collective (ReduceOp.AVG) instead of a
    second pass over the buffer."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        world = dist.get_world_size(group)
        if buf.is_cuda and scale is not None and abs(scale * world - 1.0) < 1e-12 and AVG_ON_COLLECTIVE:
            dist.all_reduce(buf, op=dist.ReduceOp.AVG, group=group)
            return buf
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    if scale is not None and scale != 1.0:
        buf.mul_(scale)
    return buf


def allgather_rows(local: torch.Tensor, out: torch.Tensor, group=None) -> torch.Tensor:
    """out[rank * k : (rank + 1) * k] = local[0:k] of every rank (k = local.shape[0]); a copy when there is one rank."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_gather_into_tensor(out, local, group=group)
    else:
        out.copy_(local)
    return out


class CapturedStep:
    """A captured SplatTrainStep.forward_backward (CUDA graph).  replay() runs it on the current stream; the duplicate count of
    the PREVIOUS replay (copied to pinned host memory by the graph) is checked against the captured buffers' capacity first -
    the graph cannot re-bin, so an overflow raises and the step has to be captured again.  The graph holds the step's buffers
    of the moment: capture again after densify_and_prune and after load_state_dict, which both replace them."""

    def __init__(self, graph, host_count, d_cap, state, outputs):
        self.graph, self._host, self.d_cap = graph, host_count, int(d_cap)
        self.state, self.outputs = state, outputs           # tensors of the graph's private pool (valid after every replay)
        self._replays = 0

    def replay(self):
        if self._replays and int(self._host[0]) > self.d_cap:
            raise RuntimeError(f"rodygs_b200: the captured step produced {int(self._host[0])} tile instances but its buffers hold "
                               f"{self.d_cap}; that frame was truncated - capture the step again")
        self._replays += 1
        self.graph.replay()


class SplatTrainStep:
    """Holds the flat parameter and gradient buffers of a static + dynamic model and runs
    forward + losses + backward for one view.

    loss = w_l1 * L1 + w_dssim * (1 - SSIM)                 (train_kubric_mrig.yaml:135-144)
         + w_pearson * (1 - Pearson(depth, gt_depth))       (:145-150, global)
         + w_local * mean_b (1 - Pearson_b)                 (:151-158, LocalPearsonDepthLoss over random box_p x box_p boxes,
                                                             losses.py:132-182; n = int(p_corr * (H // box_p) * (W // box_p)))
         + w_alpha * mean(1 - alpha)                        (benchmark-only term, SURVEY.md §8d)
    All of it is ONE loss stage (rdg_losses: three passes + a one-block finalize for the boxes).
    """

    def __init__(self, scene: Dict, height: int, width: int, sh_degree: int = 3, w_l1: float = 0.8,
                 w_dssim: float = 0.2, w_pearson: float = 0.05, w_alpha: float = 0.0, device="cuda",
                 process_group=None, w_local: float = 0.15, box_p: int = 128, p_corr: float = 0.5):
        self.dev = torch.device(device)
        self.H, self.W, self.sh_degree = int(height), int(width), int(sh_degree)
        self.w = (float(w_l1), float(w_dssim), float(w_pearson), float(w_alpha))
        # LocalPearsonDepthLoss(box_p=128, p_corr=0.5), weight 0.15 in every reference config
        self.w_local, self.box_p = float(w_local), int(box_p)
        self.n_local = int(p_corr * math.floor(self.H / self.box_p) * math.floor(self.W / self.box_p)) if w_local != 0.0 else 0
        self.pg = process_group
        self.optim: Dict[str, "GaussianAdam"] = {}
        self._skip_step = set()             # models whose next optimizer_step is the reference's post-densification no-op
        self.stats: Dict[str, "DensifyStats"] = {}
        self._load_scene(scene)
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.bg = torch.zeros(3, dtype=torch.float32, device=self.dev)          # rodygs.py:267
        self.view_grad = torch.zeros(4, 4, **f32)
        self.loss_parts = torch.zeros(8, **f32)   # [0:3] photometric (loss, l1, ssim), [3] pearson, [4] alpha term, [5] local pearson
        self._alloc_boxes()
        self.local_box_origins = None             # tests: fixed [n, 2] (row0, col0) instead of the random draw
        self.dL_dcolor = torch.empty(3, self.H, self.W, **f32)
        self.dL_ddepth = torch.zeros(1, self.H, self.W, **f32)
        self.dL_dalpha = torch.zeros(1, self.H, self.W, **f32)
        lib = _lib.load()
        self._ws_bytes = int(lib.rdg_l1_dssim_workspace_bytes(3, self.H, self.W))
        self._loss_ws = torch.empty(self._ws_bytes, dtype=torch.uint8, device=self.dev)
        self.views_per_rank = 1
        self.last_state: Optional[engine.FwdState] = None
        self._deferred = None      # exchange_grads(defer_sh=True): the factors the next optimizer_step consumes
        self.stage_events = None   # set by enable_stage_timing()

    def _alloc_boxes(self):
        if self.n_local > 0:
            # boxes (row0, col0, rows, cols): the origins are redrawn on the device every step like the reference does
            # (torch.randint(0, max_h) / (0, max_w), losses.py:149-150): one randint launch + one remainder launch
            self._boxes = torch.zeros(self.n_local, 4, dtype=torch.int32, device=self.dev)
            self._boxes[:, 2:] = self.box_p
            self._box_limits = torch.tensor([self.H - self.box_p, self.W - self.box_p], dtype=torch.int32, device=self.dev)
            self._box_rand = torch.empty(self.n_local, 2, dtype=torch.int32, device=self.dev)

    def _load_scene(self, scene: Dict):
        """(Re)build everything whose size depends on the Gaussian counts: the flat parameter / gradient buffers, the
        birth-frame CSR, the per-Gaussian scratch.  Called by __init__ and after every densification."""
        ns, nd = scene["static"]["xyz"].shape[0], scene["dynamic"]["xyz"].shape[0]
        self.ns, self.nd = ns, nd
        self.num_basis = scene["motion_coeff"].shape[-1]
        self.T = scene["table"].shape[0]
        self.layout, total = flat_layout(ns, nd, self.num_basis, self.T)
        self._set_cache = {}
        self.params = torch.zeros(total, dtype=torch.float32, device=self.dev)
        self.grads = torch.zeros(total, dtype=torch.float32, device=self.dev)
        for tag in ("static", "dynamic"):
            for k in PARAM_ORDER:
                self.p(f"{tag}.{k}").copy_(scene[tag][k])
        self.p("motion_coeff").copy_(scene["motion_coeff"])
        self.p("table").copy_(scene["table"])
        if "basis_t" in scene:                  # optional: B(t) of the last query time (checkpoints); zero otherwise
            self.p("basis_t").copy_(scene["basis_t"])
        self.time_ind = scene["time_ind"].to(self.dev, torch.int32).contiguous()
        self.spatial_lr_scale = float(scene["spatial_lr_scale"])
        self.frame_order, self.frame_offsets = engine.frame_csr(self.time_ind, self.T) if nd > 0 else (None, None)
        self._g7 = torch.empty(max(nd, 1), 8, dtype=torch.float32, device=self.dev)
        self.means2D_grad = torch.zeros(ns + nd, 3, dtype=torch.float32, device=self.dev)
        if hasattr(self, "_grads_tmp"):
            del self._grads_tmp
        self.last_state = None
        self._deferred = None      # factors of the old Gaussian set

    # -- views into the flat buffers --------------------------------------------------------
    def _slice(self, buf: torch.Tensor, name: str) -> torch.Tensor:
        off, shp = self.layout[name]
        numel = 1
        for s in shp:
            numel *= s
        return buf[off:off + numel].view(shp)

    def p(self, name: str) -> torch.Tensor:
        return self._slice(self.params, name)

    def g(self, name: str) -> torch.Tensor:
        return self._slice(self.grads, name)

    def _set(self, tag: str) -> Optional[SetArgs]:
        if (self.ns if tag == "static" else self.nd) == 0:
            return None
        # the views only change when the flat buffers are rebuilt (_load_scene): building them every step costs ~50 us
        # of host time in front of the step's first launch
        cached = self._set_cache.get(tag)
        if cached is not None and cached[0] is self.params:
            return cached[1]
        out = self._make_set(tag)
        self._set_cache[tag] = (self.params, out)
        return out

    def _make_set(self, tag: str) -> SetArgs:
        return SetArgs(xyz=self.p(f"{tag}.xyz"), scaling=self.p(f"{tag}.scaling"), rotation=self.p(f"{tag}.rotation"),
                       opacity=self.p(f"{tag}.opacity"), sh_dc=self.p(f"{tag}.features_dc"),
                       sh_rest=self.p(f"{tag}.features_rest"), sh_dc_stride=3, sh_rest_stride=45)

    def _setgrad(self, tag: str) -> SetGrads:
        if (self.ns if tag == "static" else self.nd) == 0:
            return SetGrads()
        key = ("grad", tag, self.grads.data_ptr())     # self.grads is swapped for a second buffer when accumulating
        out = self._set_cache.get(key)
        if out is None:
            out = self._make_setgrad(tag)
            self._set_cache[key] = out
        return copy.copy(out)                          # callers null some fields (factored exchange): a shallow copy

    def _make_setgrad(self, tag: str) -> SetGrads:
        return SetGrads(xyz=self.g(f"{tag}.xyz"), scaling=self.g(f"{tag}.scaling"), rotation=self.g(f"{tag}.rotation"),
                        opacity=self.g(f"{tag}.opacity"), sh_dc=self.g(f"{tag}.features_dc"),
                        sh_rest=self.g(f"{tag}.features_rest"))

    # -- timing hooks --------------------------------------------------------------------------
    def enable_stage_timing(self):
        self.stage_events = []

    def _mark(self, name: str):
        if self.stage_events is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.stage_events.append((name, ev))

    def _check_input(self, name: str, t: torch.Tensor, shape):
        if not torch.is_tensor(t) or t.dtype != torch.float32 or t.device != self.params.device or not t.is_contiguous() \
                or tuple(t.shape) != tuple(shape):
            got = f"{tuple(t.shape)} {t.dtype} {t.device} contiguous={t.is_contiguous()}" if torch.is_tensor(t) else type(t).__name__
            raise ValueError(f"SplatTrainStep: {name} must be a contiguous float32 tensor of shape {tuple(shape)} on {self.params.device}, got {got}")

    # -- one view --------------------------------------------------------------------------------
    def forward_backward(self, viewmatrix: torch.Tensor, projmatrix: torch.Tensor, tanfovx: float, tanfovy: float,
                         basis_t: torch.Tensor, gt_image: torch.Tensor, gt_depth: Optional[torch.Tensor],
                         accumulate: bool = False, forward_only: bool = False, dcolor_slot: Optional[int] = None):
        """viewmatrix / projmatrix in glm storage (V^T, P^T).  Gradients land in self.grads
        (overwritten unless accumulate=True, in which case a second flat buffer is summed in).
        dcolor_slot: data-parallel mode - do not write dL/dSH; write its 12-byte factors dL/d(rgb) into
        self.dcolor_local[dcolor_slot] instead (exchange_grads() rebuilds dL/dSH of all views from them).
        Returns self.loss_parts (device tensor; no host sync)."""
        lib = _lib.load()
        stream = _lib.stream_ptr()
        deform = self.nd > 0
        # the kernels take raw pointers: refuse anything that is not the fp32 contiguous CUDA tensor of the expected shape
        self._check_input("viewmatrix", viewmatrix, (4, 4))
        self._check_input("projmatrix", projmatrix, (4, 4))
        if deform:
            self._check_input("basis_t", basis_t, (self.num_basis, 7))
        if not forward_only:
            self._check_input("gt_image", gt_image, (3, self.H, self.W))
            if gt_depth is not None:
                self._check_input("gt_depth", gt_depth, (1, self.H, self.W))
        scene = SceneArgs(st=self._set("static"), dy=self._set("dynamic"), raw=True, use_deform=deform,
                          motion_coeff=self.p("motion_coeff").view(self.nd, self.num_basis) if deform else None,
                          time_ind=self.time_ind if deform else None, basis_t=basis_t if deform else None,
                          table=self.p("table") if deform else None, spatial_lr_scale=self.spatial_lr_scale,
                          frame_order=self.frame_order, frame_offsets=self.frame_offsets)
        view = ViewArgs(height=self.H, width=self.W, tanfovx=tanfovx, tanfovy=tanfovy, scale_modifier=1.0,
                        sh_degree=self.sh_degree, viewmatrix=viewmatrix, projmatrix=projmatrix, bg=self.bg)
        self._mark("start")
        color, depth, alpha, radii, state = engine.render_forward(scene, view, stage_hook=self._mark)
        self.last_state = state
        self.last_outputs = (color, depth, alpha, radii)
        if forward_only:
            return None
        # ---- losses + their gradients w.r.t. the rendered maps (fused kernels) ----
        w_l1, w_ds, w_p, w_a = self.w
        use_local = self.n_local > 0 and gt_depth is not None
        use_depth = (w_p != 0.0 or use_local) and gt_depth is not None
        use_alpha = w_a != 0.0
        terms = _lib.RdgLossTerms()
        if use_depth:
            terms.depth, terms.gt_depth, terms.dL_ddepth = ptr(depth), ptr(gt_depth), ptr(self.dL_ddepth)
            terms.w_pearson, terms.pearson_eps = w_p, 1e-6
        if use_local:
            if self.local_box_origins is not None:
                self._boxes[:, :2].copy_(self.local_box_origins.to(self.dev, torch.int32))
            else:
                self._box_rand.random_(0, 1 << 30)
                torch.remainder(self._box_rand, self._box_limits, out=self._boxes[:, :2])
            terms.local_boxes, terms.n_local_boxes, terms.w_local = ptr(self._boxes), self.n_local, self.w_local
        if use_alpha:
            terms.alpha, terms.dL_dalpha, terms.w_alpha = ptr(alpha), ptr(self.dL_dalpha), w_a
        # loss_parts[0:5] are written by the finalize kernel; disabled terms keep their zero
        check(lib.rdg_losses(ptr(color), ptr(gt_image), 3, self.H, self.W, w_l1, w_ds, C.byref(terms), ptr(self.loss_parts),
                             ptr(self.dL_dcolor), ptr(self._loss_ws), self._ws_bytes, stream))
        self._mark("loss")
        # ---- backward ----
        target = self.grads
        if accumulate:
            if not hasattr(self, "_grads_tmp"):
                self._grads_tmp = torch.zeros_like(self.grads)
            target = self._grads_tmp
        saved = self.grads
        self.grads = target
        try:
            self.view_grad.zero_()
            self.g("table").zero_()
            self.g("basis_t").zero_()
            gst, gdy = self._setgrad("static"), self._setgrad("dynamic")
            dcolor = None
            if dcolor_slot is not None:
                gst.sh_dc = gst.sh_rest = gdy.sh_dc = gdy.sh_rest = None
                dcolor = self.dcolor_local[dcolor_slot]
            model_hook_wanted = (dcolor_slot is not None and dcolor_slot == self.views_per_rank - 1 and self.views_per_rank == 1
                                 and getattr(self, "world_size", 1) > 1 and getattr(self, "_bucketed", False))
            dcolor_mc = 0
            if dcolor_slot is not None and self._mc_base:
                n_all = self.ns + self.nd
                block = (self._parity * self.views_per_rank * self.world_size + self._rank * self.views_per_rank + dcolor_slot)
                dcolor_mc = self._mc_base + 4 * block * n_all * 3
            grads = SceneGrads(st=gst, dy=gdy, means2D=self.means2D_grad, dcolor=dcolor, dcolor_mc=dcolor_mc,
                               dcolor_stream=self.comm_stream if dcolor_mc else None,
                               sm_queue=self._sm_queue if (model_hook_wanted and self._sm_partition) else None,
                               viewmatrix=self.view_grad,
                               motion_coeff=self.g("motion_coeff").view(self.nd, self.num_basis) if deform else None,
                               table=self.g("table") if deform else None, basis_t=self.g("basis_t") if deform else None,
                               g7_scratch=self._g7)
            hook = model_hook = None
            if dcolor_slot is not None and dcolor_slot == self.views_per_rank - 1:
                hook = self._start_gather      # the factors of every local view are final: gather them now
                if self.views_per_rank == 1 and self.world_size > 1 and self._bucketed:
                    model_hook = self._after_model   # one view per rank: each model's range is final after its own launch
            engine.render_backward(state, self.dL_dcolor, self.dL_ddepth if use_depth else None,
                                   self.dL_dalpha if use_alpha else None, grads, stage_hook=self._mark, after_blend=hook,
                                   after_model=model_hook, bwd_plan=self._bwd_plan if model_hook is not None else None)
        finally:
            self.grads = saved
        if accumulate:
            self.grads.add_(target)
        return self.loss_parts

    def capture_forward_backward(self, viewmatrix, projmatrix, tanfovx, tanfovy, basis_t, gt_image, gt_depth) -> "CapturedStep":
        """forward_backward() of one view captured as ONE CUDA graph (single-GPU step, engine.config.sync_free): ~25 kernel
        launches, the torch fills and the per-call allocations become one cudaGraphLaunch, so the GPU does not idle while
        Python enqueues the step after the user has synchronised on the previous loss.  The tensor arguments are STATIC
        buffers: copy the next view's matrices / B(t) / targets into them, then replay().  tanfovx / tanfovy are baked in
        (re-capture for a camera with other intrinsics, and after every densification: the graph holds the old buffers).
        Gradients land in self.grads, the loss in self.loss_parts."""
        if not engine.config.sync_free:
            raise RuntimeError("capture_forward_backward needs engine.config.sync_free = True (no host read inside the step)")
        if getattr(self, "world_size", 1) > 1:
            raise RuntimeError("capture_forward_backward covers the single-GPU step (the exchange runs on side streams)")
        args = (viewmatrix, projmatrix, tanfovx, tanfovy, basis_t, gt_image, gt_depth)
        for _ in range(2):                       # warm up: buffers sized, attributes set, lazy initialisation done
            self.forward_backward(*args)
        torch.cuda.synchronize()
        st = engine._cap_state(self.params.device, self.ns + self.nd)
        engine._check_pending(st)
        graph = torch.cuda.CUDAGraph()
        engine.config.capture_host = torch.zeros(2, dtype=torch.int32).pin_memory()
        engine.config.capturing = True
        try:
            with torch.cuda.graph(graph):
                self.forward_backward(*args)
        finally:
            engine.config.capturing = False
            engine.config.capture_host = None
        host, _, d_cap = st["pending"]
        st["pending"] = None
        return CapturedStep(graph, host, d_cap, self.last_state, self.last_outputs)

    def allreduce_grads(self, scale: Optional[float] = None):
        """Sum (and optionally scale) the WHOLE flat gradient buffer over the data-parallel group
        (the plain exchange; exchange_grads() is the one that scales)."""
        allreduce_flat(self.grads, scale, self.pg)

    # -- data-parallel exchange with factored SH gradients -----------------------------------------
    def enable_factored_exchange(self, views_per_rank: int, world_size: int, copy_engine_gather: bool = True,
                                 gather_streams: int = 4, bucketed: bool = True, sm_reserve: int = 16, multicast: bool = False,
                                 sm_partition: bool = True, allreduce: str = "multimem", allreduce_ctas: int = 32, bwd_parts: int = 0,
                                 bwd_order: str = "sdt", bwd_parts_static: int = 2):
        """Buffers and the side streams for exchange_grads(): the local factors [views_per_rank, N, 3], the gathered
        ones, and a communication stream on which the collectives overlap the backward kernels.

        copy_engine_gather: keep the GATHERED factors in symmetric memory (torch.distributed._symmetric_memory) and
        let every rank push its own block into all peers' buffers with plain device-to-device copies - NVLink
        through the copy engines, no SMs, so the gather really runs under the per-Gaussian backward (whose
        persistent CTAs own the whole register file; an NCCL kernel only gets in once they retire).  Falls back to
        NCCL's all-gather when symmetric memory cannot be set up.

        multicast: write the factors through the NVLink-switch multicast mapping of the gathered buffer from the kernel that
        computes them (rdg_dcolor_multicast, multimem.st) instead of pushing them with the copy engines.  Measured on 8 B200s
        (profiles/r02_timeline_n8_mc.txt): the kernel lasts 0.44 ms - every rank receives 7 x 24 MB and its stores must be
        acknowledged - and holds SMs the per-Gaussian backward needs (0.19 -> 0.43 ms), against 0.33 ms of copy-engine pushes
        that cost no SM time; off by default."""
        import torch.distributed as dist
        n = self.ns + self.nd
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.views_per_rank, self.world_size = int(views_per_rank), int(world_size)
        if self.views_per_rank * self.world_size > 16:
            raise ValueError("factored exchange: rdg_sh_grad_views stages at most 16 views per step (views_per_rank * world_size)")
        self._fx_args = (views_per_rank, world_size, copy_engine_gather, gather_streams, bucketed, sm_reserve, multicast, sm_partition,
                         allreduce, allreduce_ctas, bwd_parts, bwd_order, bwd_parts_static)
        # sm_partition: the persistent per-Gaussian kernels launch a full-machine grid whose CTAs on the reserved SMs exit at once
        # (chunk queue, RdgSceneGrad.sm_queue) instead of a smaller grid that the hardware may place on any SM
        self._sm_partition = bool(sm_partition)
        # allreduce: how the non-SH gradient range is summed over the ranks.
        #   "nccl"      torch.distributed.all_reduce (ReduceOp.AVG: a ring; NCCL has no in-switch reduction for AVG)
        #   "multimem"  (default; falls back to "nccl" without NVLS) the gradient buffer moves into symmetric memory and
        #               rdg_allreduce_multimem reduces it inside the NVLink switch (multimem.ld_reduce + multimem.st, the
        #               1 / world scale fused).  With bwd_parts > 0 the exchange is also PIPELINED: the per-Gaussian backward
        #               runs as bwd_parts launches over the dynamic model + bwd_parts_static over the static model + the dL/dtable
        #               reduction, and every piece's structure-of-arrays ranges are reduced (one launch) while the next piece is
        #               computed.  Measured: 2.76 vs 2.87 ms/step on 2 GPUs, but 3.03-3.10 vs 2.98 ms on 8 (profiles/README.md:
        #               there the NVLink ingress - 168 MB of factors + 94 MB of all-reduce per rank - is busy for the whole tail
        #               either way and the extra launches / barriers only add to it), so it is off by default
        #   "symm_op"   torch.ops.symm_mem.multimem_all_reduce_ on the same buffer + a scaling pass (library kernel, A/B)
        import torch.distributed as dist
        self._ar_mode, self._ar_ctas = "nccl", int(allreduce_ctas)
        self._grads_symm = None
        if allreduce != "nccl" and self.world_size > 1 and dist.is_initialized():
            try:
                import torch.distributed._symmetric_memory as symm_mem
                group = self.pg if self.pg is not None else dist.group.WORLD
                buf = symm_mem.empty(self.grads.numel(), dtype=torch.float32, device=self.dev)
                hdl = symm_mem.rendezvous(buf, group)
                if not int(getattr(hdl, "multicast_ptr", 0) or 0):
                    raise RuntimeError("no multicast mapping (NVLS) for the gradient buffer")
                buf.copy_(self.grads)
                self.grads = buf                      # same layout; the views are rebuilt lazily (keyed on data_ptr)
                self._grads_symm, self._ar_mode = hdl, allreduce
                self._ar_group_name = group.group_name
                self._ar_rank = dist.get_rank(group)
            except Exception as e:   # noqa: BLE001 - the fallback is the NCCL ring
                print(f"rodygs_b200: in-switch all-reduce unavailable ({type(e).__name__}: {e}); using NCCL", file=sys.stderr)
                self._ar_mode = "nccl"
        self._symm = None
        self._mc_base = 0
        v_total = self.views_per_rank * self.world_size
        self._symm = None
        self.dcolor_all = None
        if copy_engine_gather and self.world_size > 1 and dist.is_initialized():
            try:
                import torch.distributed._symmetric_memory as symm_mem
                # two gathered buffers used alternately: step k + 1 writes the other one, so no rank can overwrite factors a slower
                # peer is still reading (the all-reduce of step k + 1 cannot complete before every rank has finished step k)
                buf = symm_mem.empty(2, v_total, n, 3, dtype=torch.float32, device=self.dev)
                group = self.pg if self.pg is not None else dist.group.WORLD
                self._symm = symm_mem.rendezvous(buf, group)
                self._dc_all2 = buf
                self.dcolor_all = buf[0]
                self._rank = dist.get_rank(group)
                k = self.views_per_rank
                # NVLS: the multicast mapping of the buffer - a store to it lands in every rank's copy (rdg_dcolor_multicast)
                mc = int(getattr(self._symm, "multicast_ptr", 0) or 0)
                self._mc_base = mc if (multicast and mc) else 0
                # my block inside every peer's gathered buffer (copy-engine path, when there is no multicast mapping)
                self._peer_blocks = [[self._symm.get_buffer(r, buf.shape, torch.float32)[par, self._rank * k:(self._rank + 1) * k]
                                      for r in range(self.world_size)] for par in range(2)]
                self._gather_streams = [torch.cuda.Stream(device=self.dev) for _ in range(max(1, int(gather_streams)))]
                self._ev_push = [torch.cuda.Event() for _ in self._gather_streams]
            except Exception as e:   # noqa: BLE001 - any failure here only costs the overlap, never correctness
                print(f"rodygs_b200: symmetric-memory gather unavailable ({type(e).__name__}: {e}); using NCCL all-gather", file=sys.stderr)
                self._symm = None
                self.dcolor_all = None
        if self.dcolor_all is None:
            self._dc_all2 = torch.zeros(2, v_total, n, 3, **f32)
            self.dcolor_all = self._dc_all2[0]
            self._mc_base = 0
        self._dc_all2.zero_()
        self._parity = 0
        self.dcolor_local = torch.zeros(self.views_per_rank, n, 3, **f32)
        self.comm_stream = torch.cuda.Stream(device=self.dev)
        self.ar_stream = torch.cuda.Stream(device=self.dev)     # the all-reduces do not queue behind the gather
        self._ev_factors, self._ev_gathered = torch.cuda.Event(), torch.cuda.Event()
        self._ev_backward, self._ev_reduced = torch.cuda.Event(), torch.cuda.Event()
        self._ev_barrier = torch.cuda.Event()
        self._gather_started = False
        # bucketed all-reduce of the non-SH range: the per-Gaussian backward runs one launch per model (dynamic first) and each
        # model's range is all-reduced on the communication stream as soon as it is written - the dynamic range (xyz .. opacity,
        # motion coefficients, table) under the static model's kernel.  The persistent backward kernels leave `sm_reserve` SMs
        # to NCCL (their CTAs take the whole register file of an SM; without free SMs the collective only starts when they retire).
        self._bucketed = bool(bucketed) and self.world_size > 1 and self.ns > 0 and self.nd > 0
        self._buckets = {"static": (self.layout["static.xyz"][0], self.layout["dynamic.xyz"][0]),
                         "dynamic": (self.layout["dynamic.xyz"][0], sh_start(self.layout))}
        self._ev_piece = {}
        self._buckets_started = 0
        # pipelined exchange (in-switch all-reduce only: the pieces are structure-of-arrays slices, one launch each)
        self._bwd_plan, self._bwd_pieces, self._bwd_final = None, None, None
        if self._bucketed and self._ar_mode == "multimem" and int(bwd_parts) > 0:
            self._bwd_plan, self._bwd_pieces = self._make_bwd_plan(int(bwd_parts), bwd_order, max(1, int(bwd_parts_static)))
            self._bwd_final = [p[4] for p in self._bwd_plan if self._bwd_pieces[p[4]]][-1]
        self._sm_queue = torch.zeros(8, dtype=torch.int32, device=self.dev)
        if self._bucketed:
            _lib.set_tunable("sm_reserve", int(sm_reserve))

    def _start_gather(self):
        """All-gather of the factors on the communication stream (called right after the blend backward)."""
        self._ev_factors.record()
        with torch.cuda.stream(self.comm_stream):
            if not self._mc_base:
                self.comm_stream.wait_event(self._ev_factors)
            if self._mc_base:
                # the factors were multicast into every rank's buffer by the kernel that computed them: all that is left is the
                # cross-rank barrier that says "everybody's stores have landed"
                self._symm.barrier()
            elif self._symm is not None:
                # pushes through the copy engines on a few streams at once
                self._ev_barrier.record(self.comm_stream)
                ns = len(self._gather_streams)
                for i, st in enumerate(self._gather_streams):
                    st.wait_event(self._ev_barrier)
                    with torch.cuda.stream(st):
                        for s in range(i, self.world_size, ns):
                            r = (self._rank + s) % self.world_size
                            self._peer_blocks[self._parity][r].copy_(self.dcolor_local, non_blocking=True)
                        self._ev_push[i].record(st)
                for ev in self._ev_push:
                    self.comm_stream.wait_event(ev)
                self._symm.barrier()                    # every rank's pushes have landed everywhere
            else:
                allgather_rows(self.dcolor_local, self._dc_all2[self._parity], self.pg)
            self._ev_gathered.record(self.comm_stream)
        self._gather_started = True

    def _piece_ranges(self, tag: str, part: int, parts: int):
        """Float ranges (offset, length) inside the flat buffers of the per-Gaussian gradients that the part-th of `parts`
        launches of model `tag` writes (rdg_preprocess_bwd splits the model's 256-Gaussian chunks into equal runs)."""
        n = self.ns if tag == "static" else self.nd
        chunks = (n + 255) // 256
        per = (chunks + parts - 1) // parts
        g0, g1 = min(per * part, chunks) * 256, min(per * (part + 1), chunks) * 256
        last = g1 >= n
        g1 = min(g1, n)
        fields = [(f"{tag}.xyz", 3), (f"{tag}.scaling", 3), (f"{tag}.rotation", 4), (f"{tag}.opacity", 1)]
        if tag == "dynamic":
            fields.append(("motion_coeff", self.num_basis))
        out = []
        for name, width in fields:
            off = self.layout[name][0]
            lo, hi = off + g0 * width, off + g1 * width
            if last:
                hi = (hi + 3) // 4 * 4          # the block is padded to 64 floats (zeros on every rank)
            if hi > lo:
                out.append((lo, hi - lo))
        return out

    def _make_bwd_plan(self, parts_dynamic: int, order: str = "sdt", parts_static: int = 1):
        """Schedule of the per-Gaussian backward under the pipelined exchange: `order` is a permutation of s (static model,
        `parts_static` launches), d (dynamic model, `parts_dynamic` launches) and t (the dL/dtable reduction, after d).  The all-reduce of a
        piece starts as soon as it is written and runs under the following launches, so only the last piece's all-reduce is
        exposed; the 45 KB table range rides on the next piece's launch when there is one."""
        assert sorted(order) == ["d", "s", "t"] and order.index("d") < order.index("t"), order
        plan, pieces, carry = [], {}, []
        for ch in order:
            if ch == "d":
                for k in range(parts_dynamic):
                    name = f"dynamic.{k}"
                    plan.append((2, k, parts_dynamic, 1, name))
                    pieces[name] = self._piece_ranges("dynamic", k, parts_dynamic) + carry
                    carry = []
            elif ch == "s":
                for k in range(parts_static):
                    name = f"static.{k}"
                    plan.append((1, k, parts_static, 1, name))
                    pieces[name] = self._piece_ranges("static", k, parts_static) + carry
                    carry = []
            else:
                lo = self.layout["table"][0]
                plan.append((2, 0, 1, 2, "table"))
                if ch == order[-1]:
                    pieces["table"] = [(lo, sh_start(self.layout) - lo)]
                else:
                    pieces["table"] = []            # reduced with the next piece
                    carry = [(lo, sh_start(self.layout) - lo)]
        return tuple(plan), pieces

    def _after_model(self, piece: str):
        """Called by engine.render_backward right after the launch that completes `piece` of the per-Gaussian gradients:
        all-reduce (mean over the ranks) of that piece on the all-reduce stream."""
        ev = self._ev_piece.get(piece)
        if ev is None:
            ev = self._ev_piece[piece] = torch.cuda.Event()
        ev.record()
        with torch.cuda.stream(self.ar_stream):
            self.ar_stream.wait_event(ev)
            if self._bwd_plan is None:
                lo, hi = self._buckets[piece]
                self._allreduce_range(lo, hi)
            elif self._bwd_pieces[piece]:
                # (a piece of a model with fewer chunks than pieces is empty; the LAST piece with ranges closes the step)
                self._allreduce_ranges(self._bwd_pieces[piece], final=(piece == self._bwd_final))
        self._buckets_started += 1

    def _allreduce_ranges(self, ranges, final: bool):
        """In-switch mean over the ranks of several ranges of the symmetric gradient buffer (one launch).  The barrier in front
        says every rank has written the ranges (and, for the next call, that the previous call's slices have landed); only
        the last call of a step needs one behind it."""
        hdl = self._grads_symm
        n = len(ranges)
        offs, lens = (C.c_int64 * n)(*[r[0] for r in ranges]), (C.c_int64 * n)(*[r[1] for r in ranges])
        hdl.barrier(channel=0)
        check(_lib.load().rdg_allreduce_multimem_ranges(int(hdl.multicast_ptr), offs, lens, n, self._ar_rank, self.world_size,
                                                        1.0 / self.world_size, self._ar_ctas, _lib.stream_ptr()))
        if final:
            hdl.barrier(channel=0)

    def _allreduce_range(self, lo: int, hi: int):
        """Mean over the ranks of self.grads[lo:hi], on the current stream."""
        if self._ar_mode == "multimem":
            hdl = self._grads_symm
            hdl.barrier(channel=0)                   # every rank has written its gradients of this range
            check(_lib.load().rdg_allreduce_multimem(int(hdl.multicast_ptr) + 4 * lo, hi - lo, self._ar_rank, self.world_size,
                                                     1.0 / self.world_size, self._ar_ctas, _lib.stream_ptr()))
            hdl.barrier(channel=0)                   # every rank's slice has landed everywhere
        elif self._ar_mode == "symm_op":
            torch.ops.symm_mem.multimem_all_reduce_(self.grads[lo:hi], "sum", self._ar_group_name)
            self.grads[lo:hi].mul_(1.0 / self.world_size)
        else:
            allreduce_flat(self.grads[lo:hi], 1.0 / self.world_size, self.pg)

    def exchange_grads(self, viewmats_all: torch.Tensor, basis_all: torch.Tensor, defer_sh: bool = False):
        """Finish a data-parallel step whose local views ran with dcolor_slot=0..views_per_rank-1:
        all-gather the 12-byte factors of dL/dSH (81 % of the gradient message as 192-byte blocks; started right
        after the blend backward, so it overlaps the per-Gaussian backward), all-reduce everything else on the
        communication stream while this stream rebuilds dL/dSH of ALL views from the factors (rdg_sh_grad_views).
        viewmats_all [V,4,4] glm storage and basis_all [V,K,7] in rank-major view order (rank r holds views
        r*views_per_rank ..); the result in self.grads is the mean over the V views.

        defer_sh=True: dL/dSH is NOT materialised.  The gathered factors stay where they are and the next
        optimizer_step(tag) of each model consumes them inside the Adam update of its f_dc / f_rest groups
        (rdg_sh_adam_views: the gradient of a 256-Gaussian chunk only ever exists in shared memory), so the 384 MB
        write + re-read of the SH gradient blocks disappears from the step.  self.g("*.features_*") is then stale;
        materialize_sh_grads() rebuilds it on demand (tests, logging)."""
        lib = _lib.load()
        v_total = self.views_per_rank * self.world_size
        self._check_input("viewmats_all", viewmats_all, (v_total, 4, 4))
        if self.nd > 0:
            self._check_input("basis_all", basis_all, (v_total, self.num_basis, 7))
        n_plain = sh_start(self.layout)
        cur = torch.cuda.current_stream()
        if not self._gather_started:
            self._start_gather()
        self._gather_started = False
        if self._buckets_started == (2 if self._bwd_plan is None else len(self._bwd_plan)):
            # every range is already in flight (or done) on the communication stream
            self._buckets_started = 0
            with torch.cuda.stream(self.ar_stream):
                self._ev_reduced.record(self.ar_stream)
        else:
            self._buckets_started = 0
            self._ev_backward.record()
            with torch.cuda.stream(self.ar_stream):
                self.ar_stream.wait_event(self._ev_backward)
                self._allreduce_range(0, n_plain)
                if self.views_per_rank > 1:
                    self.grads[:n_plain].mul_(1.0 / self.views_per_rank)
                self._ev_reduced.record(self.ar_stream)
        cur.wait_event(self._ev_gathered)
        self._deferred = None
        if defer_sh:
            # the factors of this step live in _dc_all2[parity] until the step after next overwrites them
            self._deferred = {"viewmats": viewmats_all, "basis": basis_all, "dcolor": self._dc_all2[self._parity],
                              "views": v_total, "pending": {"static", "dynamic"}}
        else:
            self._sh_from_factors(viewmats_all, basis_all, self._dc_all2[self._parity], v_total,
                                  partitioned=self._bucketed and self._sm_partition)
        self._parity ^= 1
        cur.wait_event(self._ev_reduced)
        self._mark("exchange")

    def _factor_scene(self, basis_all):
        deform = self.nd > 0
        scene = SceneArgs(st=self._set("static"), dy=self._set("dynamic"), raw=True, use_deform=deform,
                          motion_coeff=self.p("motion_coeff").view(self.nd, self.num_basis) if deform else None,
                          time_ind=self.time_ind if deform else None, basis_t=basis_all[0] if deform else None,
                          table=self.p("table") if deform else None, spatial_lr_scale=self.spatial_lr_scale,
                          frame_order=self.frame_order, frame_offsets=self.frame_offsets)
        return engine._scene_struct(scene)

    def _sh_from_factors(self, viewmats_all, basis_all, dcolor_all, v_total, partitioned=False):
        sc_s = self._factor_scene(basis_all)
        gst, gdy = engine._setgrad_struct(self._setgrad("static")), engine._setgrad_struct(self._setgrad("dynamic"))
        check(_lib.load().rdg_sh_grad_views(C.byref(sc_s), self.sh_degree, v_total, ptr(viewmats_all), ptr(basis_all),
                                            ptr(dcolor_all), 1.0 / v_total, C.byref(gst), C.byref(gdy),
                                            self._sm_queue[4:].data_ptr() if partitioned else None, _lib.stream_ptr()))

    def materialize_sh_grads(self):
        """After exchange_grads(defer_sh=True): write dL/dSH of the step into self.grads after all (what exchange_grads does
        by default).  The deferred factors stay pending for the optimiser."""
        d = getattr(self, "_deferred", None)
        if d is None:
            raise RuntimeError("no deferred SH gradient: call exchange_grads(defer_sh=True) first")
        self._sh_from_factors(d["viewmats"], d["basis"], d["dcolor"], d["views"])

    def _sh_adam_from_factors(self, tag: str, iteration: int, grad_scale: float):
        """Adam of model `tag`'s f_dc / f_rest groups straight from the deferred factors (rdg_sh_adam_views)."""
        d = self._deferred
        opt = self.optim[tag]
        lr = opt.lrs.group_lrs(iteration, opt.spatial_lr_scale)
        a = _lib.RdgShAdam()
        (m_dc, v_dc), (m_rest, v_rest) = opt.moments("f_dc"), opt.moments("f_rest")
        a.exp_avg_dc, a.exp_avg_sq_dc, a.exp_avg_rest, a.exp_avg_sq_rest = ptr(m_dc), ptr(v_dc), ptr(m_rest), ptr(v_rest)
        a.lr_dc, a.lr_rest, a.step = lr["f_dc"], lr["f_rest"], opt.steps + 1
        sc_s = self._factor_scene(d["basis"])
        none = C.POINTER(_lib.RdgShAdam)()
        check(_lib.load().rdg_sh_adam_views(C.byref(sc_s), self.sh_degree, d["views"], ptr(d["viewmats"]), ptr(d["basis"]),
                                            ptr(d["dcolor"]), float(grad_scale) / d["views"],
                                            C.byref(a) if tag == "static" else none, C.byref(a) if tag == "dynamic" else none,
                                            opt.betas[0], opt.betas[1], opt.eps, _lib.stream_ptr()))

    # -- motion-basis MLP (SURVEY.md §8 a1) ----------------------------------------------------------------
    def attach_basis_mlp(self, mlp, train_times: torch.Tensor, lr: float = 1.6e-3):
        """mlp: rodygs_b200.deform.BasisMLP.  train_times [T]: the dataset's normalised frame times, whose
        embeddings the reference caches as `_time_batch_embeddings` (rodygs_dynamic.py:58-77).  After this,
        basis_forward(t) fills B(t) and the table of the flat PARAMETER buffer straight from the network and
        basis_backward() turns their gradients into the network's packed parameter gradient."""
        assert train_times.numel() == self.T, "one training time per table row"
        self.mlp = mlp
        self._mlp_times = torch.cat((torch.zeros(1), train_times.detach().float().cpu().reshape(-1))).to(self.dev)
        self._mlp_lr = float(lr)            # deform_lr_init of every reference config (train_kubric_mrig.yaml: 0.0016)
        self._mlp_moments = None
        self._mlp_steps = 0                 # Adam's own step count (bias correction), like torch.optim.Adam's state["step"]
        return mlp

    def basis_forward(self, t) -> torch.Tensor:
        """One launch: B(t) -> p("basis_t"), B(t_i) for all training times -> p("table")
        (get_gaussian_deformation + get_total_motion_table, rodygs_dynamic.py:122-147).  Returns the B(t) slice,
        which is what forward_backward(basis_t=...) takes.  t: python float or 0-d tensor (no host sync either way)."""
        if torch.is_tensor(t):
            self._mlp_times[0:1].copy_(t.reshape(1), non_blocking=True)
        else:
            self._mlp_times[0:1].fill_(float(t))
        self.mlp.forward_rows(times=self._mlp_times, out=self.p("table"), out_row0=self.p("basis_t"))
        return self.p("basis_t")

    def basis_backward(self, accumulate: bool = False) -> torch.Tensor:
        """dL/dB(t) and dL/dtable of the flat GRADIENT buffer -> mlp.grad (two launches, deterministic)."""
        return self.mlp.backward_rows(self.g("table"), d_row0=self.g("basis_t"), accumulate=accumulate)

    def allreduce_basis_grads(self, scale: Optional[float] = None):
        """Data parallel: sum the network's packed gradient (68 656 floats) over the ranks.  Call basis_backward() on the
        rank-LOCAL dL/dB(t) / dL/dtable first, i.e. before exchange_grads() / allreduce_grads(): B(t) belongs to the rank's
        own view time, so its gradient must go through the network before anything is summed across views."""
        return allreduce_flat(self.mlp.grad, scale, self.pg)

    def basis_optimizer_step(self, iteration: Optional[int] = None, grad_scale: float = 1.0):
        """Adam step of the "deform_network" group (append_motion_optim, src/trainer/rodygs_dynamic.py:101-106: one group,
        eps 1e-15) on the packed buffer - one rdg_adam launch.  The learning rate is constant = deform_lr_init:
        update_learning_rate (:199-213) looks for a group named "deform", which does not exist, so the exponential
        schedule built at :118-123 is never applied.  Bias correction uses the number of steps THIS optimiser has taken
        (torch.optim.Adam's per-parameter state["step"]), not the training iteration: the two differ whenever the network
        was not stepped from iteration 1 on (warm-up, late attach, resume).  `iteration` is accepted for call-site
        compatibility and ignored."""
        mlp = self.mlp
        self._mlp_steps += 1
        if self._mlp_moments is None:
            self._mlp_moments = (torch.zeros_like(mlp.grad), torch.zeros_like(mlp.grad))
        m, v = self._mlp_moments
        check(_lib.load().rdg_adam(ptr(mlp.params), ptr(mlp.grad), ptr(m), ptr(v), mlp.params.numel(), self._mlp_lr, 0.9, 0.999,
                                   1e-15, int(self._mlp_steps), float(grad_scale), _lib.stream_ptr()))

    # -- optimiser, densification (SURVEY.md §8 f1 / f2) ------------------------------------------------
    def _group_ranges(self, tag: str) -> Dict[str, Tuple[int, int]]:
        """reference group name -> (float offset, numel) of model `tag` inside the flat buffers."""
        from .optim import GROUP_OF
        out = {}
        for field, group in GROUP_OF.items():
            off, shp = self.layout[f"{tag}.{field}"]
            out[group] = (off, math.prod(shp))
        if tag == "dynamic":
            off, shp = self.layout["motion_coeff"]
            out["motion_coeff"] = (off, math.prod(shp))
        return out

    def attach_optimizer(self, tag: str, lrs) -> "GaussianAdam":
        """optim_setup (+ append_motion_optim for the dynamic model): rodygs_static.py:106-141, rodygs_dynamic.py:92-123."""
        from .optim import GaussianAdam
        opt = GaussianAdam(self._group_ranges(tag), self.params.numel(), lrs, self.spatial_lr_scale, self.dev)
        self.optim[tag] = opt
        return opt

    def optimizer_step(self, tag: str, iteration: int, grad_scale: float = 1.0):
        """current_gs.update_learning_rate(iteration); current_gs.optimizer.step() (rodygs.py:209,364).
        The reference densifies BEFORE optimizer.step() in the same iteration (rodygs.py:343-364); densification re-creates
        every nn.Parameter of the model, their .grad is None, and torch.optim.Adam skips them - so on a densification
        iteration that model's step is a no-op (no update, no step count).  densify_and_prune() arms the same skip here."""
        d = getattr(self, "_deferred", None)
        fused_sh = d is not None and tag in d["pending"]
        if fused_sh:
            d["pending"].discard(tag)
        if tag in self._skip_step:
            self._skip_step.discard(tag)
            return None
        if fused_sh and (self.ns if tag == "static" else self.nd) > 0:
            # exchange_grads(defer_sh=True): the SH groups step from the gathered factors - first, because the directions are
            # evaluated from the means / motion coefficients that the second launch moves
            self._sh_adam_from_factors(tag, iteration, grad_scale)
            return self.optim[tag].step(self.params, self.grads, iteration, grad_scale, skip=("f_dc", "f_rest"))
        return self.optim[tag].step(self.params, self.grads, iteration, grad_scale)

    def enable_densification(self, tag: str):
        from .densify import DensifyStats
        self.stats[tag] = DensifyStats(self.ns if tag == "static" else self.nd, self.dev)
        return self.stats[tag]

    def add_densification_stats(self, tag: str):
        """rodygs.py:319-341 after a backward pass: the radii and the means2D gradient sink of the half being trained."""
        radii = self.last_outputs[3]
        self.stats[tag].add(radii, self.means2D_grad, 0 if tag == "static" else self.ns)

    def _model_tensors(self, tag: str):
        from .optim import GROUP_OF
        params = {g: self.p(f"{tag}.{f}") for f, g in GROUP_OF.items()}
        if tag == "dynamic":
            params["motion_coeff"] = self.p("motion_coeff")
        return params

    def densify_and_prune(self, tag: str, grad_threshold: float, min_opacity: float, extent: float,
                          max_screen_size: Optional[float], percent_dense: float = 0.01, noise=None, generator=None):
        """current_gs.densify_and_prune(...) (rodygs.py:343-356) on model `tag`; the flat buffers, the optimiser
        moments, the statistics and the birth-frame table are rebuilt for the new Gaussian count.  Under data
        parallelism every rank calls this with all-reduced statistics and the same noise."""
        from . import densify as dn
        from .optim import GROUP_OF
        if tag in self.stats:
            # every data-parallel user of this class runs on the default group (process_group=None): the statistics must be
            # made rank-consistent there too, or the ranks clone / split / prune different rows and their buffer sizes
            # diverge.  all_reduce() is a no-op for a single process.
            self.stats[tag].all_reduce(self.pg)
        params = self._model_tensors(tag)
        opt = self.optim.get(tag)
        moments = {g: opt.moments(g) for g in params} if opt is not None else None
        moments = {g: (m.view(params[g].shape), v.view(params[g].shape)) for g, (m, v) in moments.items()} if moments else None
        extras = {"time_ind": self.time_ind} if tag == "dynamic" else None
        new_p, new_m, new_e, new_stats, info = dn.densify_and_prune(params, moments, extras, self.stats[tag], grad_threshold,
                                                                    min_opacity, extent, max_screen_size, percent_dense,
                                                                    noise=noise, generator=generator)
        other = "dynamic" if tag == "static" else "static"
        inv = {g: f for f, g in GROUP_OF.items()}
        scene = {tag: {inv[g]: t for g, t in new_p.items() if g in inv},
                 other: {k: self.p(f"{other}.{k}") for k in PARAM_ORDER},
                 "motion_coeff": new_p["motion_coeff"] if tag == "dynamic" else self.p("motion_coeff"),
                 "table": self.p("table"), "time_ind": new_e["time_ind"] if tag == "dynamic" else self.time_ind,
                 "spatial_lr_scale": self.spatial_lr_scale}
        old_moments = {}
        for t, o in self.optim.items():
            old_moments[t] = {g: o.moments(g) for g in o.ranges} if t != tag else \
                {g: (m.reshape(-1), v.reshape(-1)) for g, (m, v) in new_m.items()}
        old_stats = {t: st for t, st in self.stats.items() if t != tag}
        self._load_scene(scene)
        from .optim import GaussianAdam
        for t, o in list(self.optim.items()):
            fresh = GaussianAdam(self._group_ranges(t), self.params.numel(), o.lrs, self.spatial_lr_scale, self.dev, o.betas, o.eps)
            fresh.steps = o.steps
            for g, (m, v) in old_moments[t].items():
                fm, fv = fresh.moments(g)
                fm.copy_(m)
                fv.copy_(v)
            self.optim[t] = fresh
        self.stats = dict(old_stats)
        self.stats[tag] = new_stats
        if getattr(self, "_fx_args", None) is not None:          # the exchange buffers are sized by the Gaussian count
            self.enable_factored_exchange(*self._fx_args)
        if tag in self.optim:
            self._skip_step.add(tag)
        return info

    def reset_opacity(self, tag: str, cap: float = 0.01):
        """current_gs.reset_opacity() (rodygs.py:358-362)."""
        from . import densify as dn
        opt = self.optim.get(tag)
        dn.reset_opacity(self.p(f"{tag}.opacity"), opt.moments("opacity") if opt is not None else None, cap)

    # -- motion regularisers (SURVEY.md §8 f4) --------------------------------------------------------
    def motion_losses_backward(self, iteration: int, basis_t: torch.Tensor, w_motion_l1: float = 0.01,
                               w_sparsity: float = 0.002, w_basis: float = 0.1, basis_mode: str = "cum_exponential",
                               w_rigidity: float = 0.5, rigidity_freq: int = 5, K: int = 8, sample_scale: float = 2,
                               dist_preserving_ratio: int = 4, indice: Optional[torch.Tensor] = None,
                               frame_indices: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The dynamic model's regularisers of configs/train/*.yaml:198-237 (motion_l1_reg, motion_sparsity, rigidity
        with freq 5, motion_basis_reg), each gated like MultiLoss.forward (losses.py:67-73: `iteration % freq == 0 and
        iteration > start`, start 0), value + gradient in one C-ABI call each; the weighted gradients are ADDED to the
        flat gradient buffer that forward_backward() has just written.  Returns motion_parts [6] on the device:
        (mean|c|, sparsity, basis translation, basis rotation, rigidity surface, rigidity distance-preserving).
        indice / frame_indices override the reference's random draws (tests)."""
        from . import motion_reg as mr
        import random
        lib = _lib.load()
        stream = _lib.stream_ptr()
        parts = torch.zeros(6, dtype=torch.float32, device=self.dev)
        if self.nd == 0 or iteration <= 0:
            return parts
        coeff = self.p("motion_coeff").view(self.nd, self.num_basis)
        d_coeff = self.g("motion_coeff").view(self.nd, self.num_basis)
        table, d_table = self.p("table"), self.g("table")
        if w_motion_l1 != 0.0 or w_sparsity != 0.0:
            parts[0:2] = mr.motion_coeff_reg_(coeff, w_motion_l1, w_sparsity, d_coeff, accumulate=True)
        if w_basis != 0.0:
            if getattr(self, "_basis_mode", None) != basis_mode:
                self._basis_mode, self._basis_reg = basis_mode, mr.basis_reg_coeff(basis_mode).to(self.dev)
            parts[2:4] = mr.motion_basis_reg_(table, self._basis_reg, 0, 0, d_table, grad_scale=w_basis)
        if w_rigidity != 0.0 and iteration % rigidity_freq == 0:
            scale = 1 / sample_scale if sample_scale > 1 else sample_scale
            if indice is None:
                indice = torch.tensor(random.sample(range(self.nd), int(self.nd * scale)))       # losses.py:228-232
            if frame_indices is None:
                frame_indices = torch.randint(0, self.T - 1, (self.T // dist_preserving_ratio,))   # :297-301
            idx = indice.to(self.dev, torch.int32).contiguous()
            fi = frame_indices.to(self.dev, torch.int32).contiguous()
            n = idx.numel()
            f32 = dict(dtype=torch.float32, device=self.dev)
            pts, canon, cs = torch.empty(n, 3, **f32), torch.empty(n, 3, **f32), torch.empty(n, self.num_basis, **f32)
            xyz = self.p("dynamic.xyz")
            check(lib.rdg_rigidity_sample(n, self.num_basis, ptr(idx), ptr(xyz), ptr(coeff), ptr(self.time_ind), ptr(basis_t),
                                          ptr(table), self.spatial_lr_scale, ptr(pts), ptr(canon), ptr(cs), stream))
            d2, nn = mr.knn_points(pts, K)
            a = _lib.RdgRigidity()
            a.n, a.K, a.num_basis, a.n_frames, a.eps = n, K, self.num_basis, fi.numel(), 1e-6
            a.mode_surface, a.mode_distance = 1, 1
            d_pts, d_canon, d_cs = torch.empty_like(pts), torch.empty_like(canon), torch.empty_like(cs)
            d_tab = torch.zeros_like(table) if w_rigidity != 1.0 else d_table
            a.points, a.canon, a.coeff, a.table, a.frame_indices = ptr(pts), ptr(canon), ptr(cs), ptr(table), ptr(fi)
            a.nn_idx, a.nn_dist2, a.loss_parts = ptr(nn), ptr(d2), parts[4:6].data_ptr()
            a.d_points, a.d_canon, a.d_coeff, a.d_table = ptr(d_pts), ptr(d_canon), ptr(d_cs), ptr(d_tab)
            nbytes = int(lib.rdg_rigidity_workspace_bytes(n, K, fi.numel()))
            ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=self.dev)
            check(lib.rdg_rigidity(C.byref(a), ptr(ws), nbytes, stream))
            if d_tab is not d_table:
                d_table.add_(d_tab, alpha=w_rigidity)
            check(lib.rdg_rigidity_sample_bwd(n, self.num_basis, self.T, ptr(idx), ptr(coeff), ptr(self.time_ind), ptr(basis_t),
                                              ptr(table), self.spatial_lr_scale, float(w_rigidity), ptr(d_pts), ptr(d_canon),
                                              ptr(d_cs), ptr(self.g("dynamic.xyz")), ptr(d_coeff), ptr(self.g("basis_t")),
                                              ptr(d_table), stream))
        self.motion_parts = parts
        return parts

    def total_loss(self) -> torch.Tensor:
        """photometric + w_p * pearson + w_local * local pearson + alpha term (device scalar)."""
        lp = self.loss_parts
        return lp[0] + self.w[2] * lp[3] + lp[4] + (self.w_local * lp[5] if self.n_local > 0 else 0.0)

    # -- checkpoints -------------------------------------------------------------------------------------------
    def _check_saveable(self):
        d = getattr(self, "_deferred", None)
        if d is not None and d["pending"]:
            raise RuntimeError("SplatTrainStep.state_dict: exchange_grads(defer_sh=True) left the SH gradient factors of "
                               f"{sorted(d['pending'])} pending; call optimizer_step for them first")

    def _dp_rank_world(self) -> Tuple[int, int]:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.pg) > 1:
            return dist.get_rank(self.pg), dist.get_world_size(self.pg)
        return 0, 1

    def _rank_state(self) -> Dict:
        """The part of the state that differs between data-parallel ranks: the densification statistics (each rank adds
        its own views' radii and means2D gradients; they are only reduced inside densify_and_prune) and the CUDA
        generator (seeded per rank)."""
        return {"stats": {tag: {f: getattr(st, f).detach().to("cpu", copy=True) for f in STATS_FIELDS}
                          for tag, st in self.stats.items()},
                "cuda_rng_state": torch.cuda.get_rng_state(self.dev)}

    def state_dict(self) -> Dict:
        """Everything a resumed run needs to train on exactly as this one would, as CPU tensors, numbers, strings, lists
        and dicts (so torch.load(weights_only=True) reads it back).  Parameters and moments are stored by name, never as
        the flat buffer: the flat layout changes with every densification.  Gradients are not state (every step
        rewrites them): save between iterations, after optimizer_step.  "ranks" holds one entry per data-parallel rank
        (statistics, CUDA generator; see _rank_state); state_dict() fills in the calling process only, save() all ranks."""
        self._check_saveable()
        from .optim import GROUP_OF
        from dataclasses import asdict

        def cpu(t):
            return t.detach().to("cpu", copy=True)

        w_l1, w_dssim, w_pearson, w_alpha = self.w
        sd = {"format": CHECKPOINT_FORMAT, "version": CHECKPOINT_VERSION,
              "ns": self.ns, "nd": self.nd, "num_basis": self.num_basis, "T": self.T, "H": self.H, "W": self.W,
              "sh_degree": self.sh_degree, "w_l1": w_l1, "w_dssim": w_dssim, "w_pearson": w_pearson, "w_alpha": w_alpha,
              "w_local": self.w_local, "box_p": self.box_p, "n_local": self.n_local,
              "params": {name: cpu(self.p(name)) for name in self.layout},
              "time_ind": cpu(self.time_ind), "spatial_lr_scale": self.spatial_lr_scale,
              "optim": {}, "skip_step": sorted(self._skip_step), "ranks": [self._rank_state()]}
        field_of = {g: f for f, g in GROUP_OF.items()}
        for tag, opt in self.optim.items():
            shapes = {g: self.layout["motion_coeff" if g == "motion_coeff" else f"{tag}.{field_of[g]}"][1] for g in opt.ranges}
            moments = {g: opt.moments(g) for g in opt.ranges}
            sd["optim"][tag] = {"lrs": {k: v for k, v in asdict(opt.lrs).items() if v is not None},
                                "betas": [float(b) for b in opt.betas], "eps": float(opt.eps), "steps": int(opt.steps),
                                "exp_avg": {g: cpu(m.view(shapes[g])) for g, (m, _) in moments.items()},
                                "exp_avg_sq": {g: cpu(v.view(shapes[g])) for g, (_, v) in moments.items()}}
        mlp = getattr(self, "mlp", None)
        if mlp is not None:
            sd["mlp"] = {"args": dict(mlp.init_args), "state_dict": {k: cpu(v) for k, v in mlp.state_dict().items()},
                         "lr": self._mlp_lr, "steps": int(self._mlp_steps), "train_times": cpu(self._mlp_times[1:])}
            if self._mlp_moments is not None:
                sd["mlp"]["exp_avg"], sd["mlp"]["exp_avg_sq"] = (cpu(t) for t in self._mlp_moments)
        return sd

    def _rank_entry(self, ranks: List[Dict]) -> Tuple[Dict, torch.Tensor]:
        """(statistics, generator state) this process resumes from.  Same number of ranks as saved: its own entry.
        Otherwise the statistics are combined (sum, sum, max) into rank 0 and the other ranks start their sums at zero, so
        the all-reduce inside the next densify_and_prune still sees every saved contribution once; rank r takes the
        generator of saved rank r mod the saved count."""
        rank, world = self._dp_rank_world()
        if len(ranks) == world:
            return ranks[rank]["stats"], ranks[rank]["cuda_rng_state"]
        stats = {}
        for tag in ranks[0]["stats"]:
            per = [r["stats"][tag] for r in ranks]
            s = {"grad_accum": sum(p["grad_accum"] for p in per), "denom": sum(p["denom"] for p in per),
                 "max_radii2D": torch.stack([p["max_radii2D"] for p in per]).amax(0)}
            if rank > 0:
                s["grad_accum"], s["denom"] = torch.zeros_like(s["grad_accum"]), torch.zeros_like(s["denom"])
            stats[tag] = s
        return stats, ranks[rank % len(ranks)]["cuda_rng_state"]

    def _parse_state(self, sd: Dict):
        """Every check of load_state_dict, before anything of this step changes."""
        from .optim import GROUP_OF, GaussianLRs
        pre = "SplatTrainStep.load_state_dict"
        for field, have in (("H", self.H), ("W", self.W)):
            if int(sd[field]) != have:
                raise ValueError(f"{pre}: {field} is {sd[field]} in the state dict but {have} here "
                                 "(the image buffers are sized by it); build the step with from_state_dict instead")
        ns, nd, K, T = (int(sd[k]) for k in ("ns", "nd", "num_basis", "T"))
        mlp = getattr(self, "mlp", None)
        if mlp is not None:
            for field, have in (("num_basis", mlp.num_basis), ("T", self._mlp_times.numel() - 1)):
                if int(sd[field]) != have:
                    raise ValueError(f"{pre}: {field} is {sd[field]} in the state dict but the attached basis MLP has {have}")
            if "mlp" not in sd:
                raise ValueError(f"{pre}: the state dict has no basis MLP but one is attached to this step (its next "
                                 "basis_forward would overwrite the saved table); load it with from_state_dict")
            for k, v in sd["mlp"]["args"].items():
                if mlp.init_args[k] != v:
                    raise ValueError(f"{pre}: the attached basis MLP has {k}={mlp.init_args[k]!r}, the state dict {v!r}")
        layout, _ = flat_layout(ns, nd, K, T)
        P = sd["params"]
        for name, (_, shp) in layout.items():
            if tuple(P[name].shape) != shp:
                raise ValueError(f"{pre}: params[{name!r}] has shape {tuple(P[name].shape)}, the saved counts give {shp}")
        if tuple(sd["time_ind"].shape) != (nd,):
            raise ValueError(f"{pre}: time_ind has shape {tuple(sd['time_ind'].shape)}, expected ({nd},)")
        scene = {tag: {k: P[f"{tag}.{k}"] for k in PARAM_ORDER} for tag in ("static", "dynamic")}
        scene.update(motion_coeff=P["motion_coeff"], table=P["table"], basis_t=P["basis_t"], time_ind=sd["time_ind"],
                     spatial_lr_scale=float(sd["spatial_lr_scale"]))
        optims = {}
        for tag, o in sd["optim"].items():
            if tag not in ("static", "dynamic"):
                raise ValueError(f"{pre}: optimiser of unknown model {tag!r}")
            groups = {g: layout[f"{tag}.{f}"][1] for f, g in GROUP_OF.items()}
            if tag == "dynamic":
                groups["motion_coeff"] = layout["motion_coeff"][1]
            for kind in ("exp_avg", "exp_avg_sq"):
                for g, shp in groups.items():
                    if o[kind][g].numel() != math.prod(shp):
                        raise ValueError(f"{pre}: optim[{tag!r}][{kind!r}][{g!r}] has {o[kind][g].numel()} elements, "
                                         f"expected {math.prod(shp)}")
            optims[tag] = (GaussianLRs(**o["lrs"]), tuple(float(b) for b in o["betas"]), float(o["eps"]), int(o["steps"]), o)
        stats, rng = self._rank_entry(sd["ranks"])
        for tag, s in stats.items():
            n = {"static": ns, "dynamic": nd}[tag]
            for f in STATS_FIELDS:
                if tuple(s[f].shape) != (n,):
                    raise ValueError(f"{pre}: statistics {tag}.{f} have shape {tuple(s[f].shape)}, expected ({n},)")
        if "mlp" in sd:
            m = sd["mlp"]
            if m["train_times"].numel() != T:
                raise ValueError(f"{pre}: the basis MLP has {m['train_times'].numel()} training times, the table {T} rows")
            missing = [k for k in ("args", "state_dict", "lr", "steps") if k not in m]
            if missing:
                raise ValueError(f"{pre}: the basis MLP entry has no {missing}")
        return scene, optims, stats, rng

    def load_state_dict(self, sd: Dict):
        """Restore a state_dict(): the flat buffers are rebuilt at the saved Gaussian counts (this step may have been built
        for any other N), then the loss configuration, the optimisers, the pending post-densification skips, the
        densification statistics, the basis MLP (built from the saved arguments when none is attached) and the CUDA
        generator that draws the local Pearson boxes.  Every check runs before anything changes; it refuses what it cannot
        repair, naming the field: another image size, a num_basis / T / network that differs from the MLP attached to this
        step, or a state without an MLP while one is attached.  Like densify_and_prune this replaces every buffer: a
        CapturedStep taken before must be captured again, and an enabled factored exchange is set up again."""
        pre = "SplatTrainStep.load_state_dict"
        if not isinstance(sd, dict) or sd.get("format") != CHECKPOINT_FORMAT or sd.get("version") != CHECKPOINT_VERSION:
            got = (sd.get("format"), sd.get("version")) if isinstance(sd, dict) else type(sd).__name__
            raise ValueError(f"{pre}: not a {CHECKPOINT_FORMAT} v{CHECKPOINT_VERSION} state dict ({got!r})")
        try:
            scene, optims, stats, rng = self._parse_state(sd)
        except (KeyError, TypeError, AttributeError) as e:
            raise ValueError(f"{pre}: malformed state dict ({type(e).__name__}: {e})") from None
        from .densify import DensifyStats
        from .optim import GaussianAdam
        self._load_scene(scene)
        self.sh_degree = int(sd["sh_degree"])
        self.w = tuple(float(sd[k]) for k in ("w_l1", "w_dssim", "w_pearson", "w_alpha"))
        self.w_local, self.box_p, self.n_local = float(sd["w_local"]), int(sd["box_p"]), int(sd["n_local"])
        self._alloc_boxes()
        self.optim = {}
        for tag, (lrs, betas, eps, steps, o) in optims.items():
            opt = GaussianAdam(self._group_ranges(tag), self.params.numel(), lrs, self.spatial_lr_scale, self.dev, betas, eps)
            opt.steps = steps
            for g in opt.ranges:
                m, v = opt.moments(g)
                m.copy_(o["exp_avg"][g].reshape(-1))
                v.copy_(o["exp_avg_sq"][g].reshape(-1))
            self.optim[tag] = opt
        self._skip_step = set(sd["skip_step"])
        self.stats = {}
        for tag, s in stats.items():
            st = DensifyStats(s["denom"].shape[0], self.dev)
            for f in STATS_FIELDS:
                getattr(st, f).copy_(s[f])
            self.stats[tag] = st
        if "mlp" in sd:
            m = sd["mlp"]
            mlp = getattr(self, "mlp", None)
            if mlp is None:
                from .deform import BasisMLP
                mlp = BasisMLP(**m["args"], device=self.dev)
            mlp.load_state_dict(m["state_dict"])
            self.attach_basis_mlp(mlp, m["train_times"], lr=float(m["lr"]))
            self._mlp_steps = int(m["steps"])
            if "exp_avg" in m:
                self._mlp_moments = (m["exp_avg"].to(self.dev), m["exp_avg_sq"].to(self.dev))
        torch.cuda.set_rng_state(rng, self.dev)
        if getattr(self, "_fx_args", None) is not None:          # the exchange buffers are sized by the Gaussian count
            self.enable_factored_exchange(*self._fx_args)
        return self

    @classmethod
    def from_state_dict(cls, sd: Dict, device="cuda", process_group=None) -> "SplatTrainStep":
        """A step built from a state_dict() alone (no scene dict): image size, loss weights and counts come from it."""
        f32 = dict(dtype=torch.float32)
        K, T = int(sd["num_basis"]), int(sd["T"])
        empty = {k: torch.zeros((0,) + s, **f32) for k, s in (("xyz", (3,)), ("scaling", (3,)), ("rotation", (4,)),
                                                             ("opacity", (1,)), ("features_dc", (1, 3)), ("features_rest", (15, 3)))}
        scene = {"static": empty, "dynamic": empty, "motion_coeff": torch.zeros(0, 1, K, **f32),
                 "table": torch.zeros(T, K, 7, **f32), "time_ind": torch.zeros(0, dtype=torch.int32), "spatial_lr_scale": 1.0}
        step = cls(scene, int(sd["H"]), int(sd["W"]), sh_degree=int(sd["sh_degree"]), device=device, process_group=process_group,
                   w_local=float(sd["w_local"]), box_p=int(sd["box_p"]))
        return step.load_state_dict(sd)

    def save(self, path):
        """torch.save(state_dict(), path).  Under data parallelism every rank calls it: the per-rank part of the state
        (_rank_state) is gathered from all ranks, rank 0 writes the file, and every rank returns once it is complete - or
        raises, on every rank, when the state cannot be saved or rank 0 could not write it."""
        import torch.distributed as dist
        self._check_saveable()                 # on every rank before any collective (the ranks hold the same pending set)
        rank, world = self._dp_rank_world()
        if world == 1:
            torch.save(self.state_dict(), path)
            return
        ranks = [None] * world
        dist.all_gather_object(ranks, self._rank_state(), group=self.pg)
        err = None
        if rank == 0:
            try:
                sd = self.state_dict()
                sd["ranks"] = ranks
                torch.save(sd, path)
            except Exception as e:   # noqa: BLE001 - reported on every rank below
                err = e
        flag = torch.tensor([0 if err is None else 1], dtype=torch.int32, device=self.dev)
        dist.broadcast(flag, 0 if self.pg is None else dist.get_global_rank(self.pg, 0), group=self.pg)
        if err is not None:
            raise err
        if int(flag.item()):
            raise RuntimeError(f"SplatTrainStep.save: rank 0 could not write {path} (see its error)")

    def load(self, path):
        """load_state_dict(torch.load(path, weights_only=True)); every rank of a data-parallel run reads the same file and
        takes its own statistics and generator from it."""
        return self.load_state_dict(torch.load(path, map_location="cpu", weights_only=True))
