"""Test-time pose refinement of held-out cameras: the reference's PoseOptimizer (RoDyGSEvaluator.eval with alignment) on the
device.  For each view, `iters` iterations of: render the static model at V(q, T), L2 photometric loss against the ground
truth, backward to dL/dV, one Adam step on (q, T).  One iteration is ONE captured CUDA graph of eight C-ABI calls
(rdg_preprocess_fwd -> rdg_bin_tiles -> rdg_blend_fwd -> rdg_l2_loss -> zero acc -> rdg_blend_bwd -> rdg_preprocess_bwd ->
rdg_pose_adam); the loop replays it in chunks with one host read per chunk.  Definitions: INTEGRATION.md "Refining held-out
camera poses".

Nothing here touches the training state: every buffer is the loop's own (the duplicate capacity of engine._capacity and a
pending sync-free count included).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Sequence, Tuple, Union

import torch

from . import _lib, engine
from ._lib import RdgBins, RdgPoseAdam, RdgSceneGrad, check, ptr
from .engine import NACC, SceneArgs, SetArgs, ViewArgs

BETAS = (0.9, 0.999)            # torch.optim.Adam defaults
EPS = 1e-8
ORTHONORMAL_TOL = 1e-4
CHUNK = 100                     # graph replays between two host reads of the step counter and the overflow latch
STATIC_FIELDS = {"xyz": (3,), "features_dc": (1, 3), "features_rest": (15, 3), "scaling": (3,), "rotation": (4,),
                 "opacity": (1,)}


def per_view(name: str, v, n_views: int) -> List[float]:
    """A float, or one float per view, as a list of n_views floats."""
    vals = [float(t) for t in v] if hasattr(v, "__len__") else [float(v)] * n_views
    if len(vals) != n_views:
        raise ValueError(f"refine_poses: {name} must be a float or {n_views} values, got {len(vals)}")
    return vals


def pose_from_viewmatrix(viewmats: torch.Tensor) -> torch.Tensor:
    """[V, 7] float32 (q_r, q_x, q_y, q_z, T) of [V, 4, 4] glm-storage view matrices, computed on their device in float64:
    q the camera-to-world rotation (unit norm, q_r >= 0), T the camera-to-world translation.  Raises ValueError naming the
    first view whose rotation block is not orthonormal to 1e-4 (or is a reflection)."""
    vm = viewmats.double()
    R = vm[:, :3, :3]                      # glm storage holds V^T: its row-major 3x3 block is R_c2w itself
    t = vm[:, 3, :3]                       # the world->view translation -R^T T
    eye = torch.eye(3, dtype=torch.float64, device=vm.device)
    err = (R @ R.transpose(1, 2) - eye).abs().amax((1, 2))
    det = torch.linalg.det(R)
    bad = ((err > ORTHONORMAL_TOL) | (det <= 0) | ~torch.isfinite(err)).nonzero()
    if bad.numel():
        v = int(bad[0, 0])
        raise ValueError(f"refine_poses: view {v}: the rotation block of viewmats[{v}] is not orthonormal to "
                         f"{ORTHONORMAL_TOL} (max |R R^T - I| = {float(err[v]):.3g}, det = {float(det[v]):.3g})")
    T = -(R @ t.unsqueeze(-1)).squeeze(-1)
    m = R
    m00, m01, m02 = m[:, 0, 0], m[:, 0, 1], m[:, 0, 2]
    m10, m11, m12 = m[:, 1, 0], m[:, 1, 1], m[:, 1, 2]
    m20, m21, m22 = m[:, 2, 0], m[:, 2, 1], m[:, 2, 2]
    # the four candidates of the matrix -> quaternion inversion; the one with the largest |component| is well conditioned
    q_abs = torch.stack([1 + m00 + m11 + m22, 1 + m00 - m11 - m22, 1 - m00 + m11 - m22, 1 - m00 - m11 + m22], -1)
    q_abs = q_abs.clamp_min(0).sqrt()
    cand = torch.stack([
        torch.stack([q_abs[:, 0] ** 2, m21 - m12, m02 - m20, m10 - m01], -1),
        torch.stack([m21 - m12, q_abs[:, 1] ** 2, m10 + m01, m02 + m20], -1),
        torch.stack([m02 - m20, m10 + m01, q_abs[:, 2] ** 2, m12 + m21], -1),
        torch.stack([m10 - m01, m20 + m02, m21 + m12, q_abs[:, 3] ** 2], -1)], 1)
    cand = cand / (2.0 * q_abs.clamp_min(0.1)).unsqueeze(-1)
    q = cand[torch.arange(vm.shape[0], device=vm.device), q_abs.argmax(-1)]
    q = q / q.norm(dim=-1, keepdim=True)
    q = torch.where(q[:, :1] < 0, -q, q)
    return torch.cat([q, T], -1).float()


def _static_set(static: Dict[str, torch.Tensor]) -> SetArgs:
    """SetArgs of the raw static model; keys are GaussianParams names, with or without the reference's leading '_'."""
    t = {}
    for name in STATIC_FIELDS:
        x = static.get(name, static.get("_" + name))
        if not torch.is_tensor(x):
            raise ValueError(f"refine_poses: static['{name}'] is missing")
        t[name] = x
    n = t["xyz"].shape[0] if t["xyz"].dim() == 2 else -1
    if n < 1:
        raise ValueError("refine_poses: the static model must have at least one Gaussian ([n, 3] xyz)")
    for name, x in t.items():
        want = (n,) + STATIC_FIELDS[name]
        if x.dtype != torch.float32 or not x.is_cuda or not x.is_contiguous() or tuple(x.shape) != want:
            raise ValueError(f"refine_poses: static['{name}'] must be a contiguous float32 CUDA tensor of shape {want}, got "
                             f"{tuple(x.shape)} {x.dtype} {x.device} contiguous={x.is_contiguous()}")
    return SetArgs(xyz=t["xyz"], scaling=t["scaling"], rotation=t["rotation"], opacity=t["opacity"], sh_dc=t["features_dc"],
                   sh_rest=t["features_rest"], sh_dc_stride=3, sh_rest_stride=45)


def _check(name: str, t, shape, dev):
    if not torch.is_tensor(t) or t.dtype != torch.float32 or t.device != dev or not t.is_contiguous() or tuple(t.shape) != tuple(shape):
        got = f"{tuple(t.shape)} {t.dtype} {t.device} contiguous={t.is_contiguous()}" if torch.is_tensor(t) else type(t).__name__
        raise ValueError(f"refine_poses: {name} must be a contiguous float32 tensor of shape {tuple(shape)} on {dev}, got {got}")


class _PoseLoop:
    """The buffers and the captured iteration of one view."""

    def __init__(self, st: SetArgs, view: ViewArgs, gt: torch.Tensor, pose0: torch.Tensor, lr: float, iters: int):
        self.lib = _lib.load()
        dev = gt.device
        self.n, self.H, self.W, self.iters = st.n(), view.height, view.width, iters
        self.tiles = engine.tiles_of(self.H, self.W)
        f32 = dict(dtype=torch.float32, device=dev)
        i32 = dict(dtype=torch.int32, device=dev)
        n, H, W = self.n, self.H, self.W
        self.scene = engine._scene_struct(SceneArgs(st=st, raw=True))
        self.geom = {"radii": torch.empty(n, **i32), "tiles_touched": torch.empty(n, **i32), "p0": torch.empty(n, 4, **f32),
                     "p1": torch.empty(n, 4, **f32), "p2": torch.empty(n, 2, **f32),
                     "clamped": torch.empty(n, dtype=torch.uint8, device=dev), "tile_count": torch.empty(self.tiles + 1, **i32)}
        self.geom_s = engine._geom_struct(self.geom)
        self.ranges = torch.empty(self.tiles, 2, **i32)
        self.num_rendered = torch.zeros(2, **i32)
        self.region_count = torch.empty(2 * self.tiles, **i32)
        self.color, self.depth, self.alpha = torch.empty(3, H, W, **f32), torch.empty(1, H, W, **f32), torch.empty(1, H, W, **f32)
        self.final_T, self.n_contrib = torch.empty(H, W, **f32), torch.empty(H, W, **i32)
        self.gt, self.dL_dcolor = gt, torch.empty(3, H, W, **f32)
        self.acc = torch.zeros(n, NACC, **f32)
        self.det_bytes = int(self.lib.rdg_blend_bwd_deterministic_scratch_bytes(n)) if engine.config.deterministic else 0
        self.det_scratch = torch.empty(self.det_bytes, dtype=torch.uint8, device=dev) if self.det_bytes else None
        self.loss_bytes = int(self.lib.rdg_l2_loss_workspace_bytes(3, H, W))
        self.loss_ws = torch.empty(self.loss_bytes, dtype=torch.uint8, device=dev)
        self.history = torch.zeros(iters, **f32)
        # pose state: (q, T), Adam moments, step counter, dL/dV, V(q, T), overflow latch
        self.pose0 = pose0
        self.param = pose0.clone()
        self.exp_avg, self.exp_avg_sq = torch.zeros(7, **f32), torch.zeros(7, **f32)
        self.step = torch.zeros(1, **i32)
        self.dV = torch.zeros(16, **f32)
        self.vm = torch.empty(16, **f32)
        self.overflow = torch.zeros(2, **i32)
        self.view = ViewArgs(height=H, width=W, tanfovx=view.tanfovx, tanfovy=view.tanfovy, scale_modifier=1.0,
                             sh_degree=view.sh_degree, viewmatrix=self.vm, projmatrix=view.projmatrix, bg=view.bg)
        self.view_s = engine._view_struct(self.view)
        self.adam = RdgPoseAdam(param=ptr(self.param), exp_avg=ptr(self.exp_avg), exp_avg_sq=ptr(self.exp_avg_sq),
                                step=ptr(self.step), dL_dV=ptr(self.dV), viewmatrix=ptr(self.vm), grad=None,
                                num_rendered=ptr(self.num_rendered), overflow=ptr(self.overflow), lr=float(lr), beta1=BETAS[0],
                                beta2=BETAS[1], eps=EPS, max_steps=iters)
        self.grads = RdgSceneGrad()                  # every pointer NULL but dL/dV: rdg_preprocess_bwd writes nothing else
        self.grads.viewmatrix = ptr(self.dV)
        self.graph = None

    def _alloc_bins(self, cap: int):
        dev = self.gt.device
        self.cap = int(cap)
        self.vals = torch.empty(self.cap, dtype=torch.int32, device=dev)
        self.region_ids = torch.empty(2 * self.cap, dtype=torch.int32, device=dev)
        self.region_masks = torch.empty(2 * self.cap, dtype=torch.uint8, device=dev)
        self.bin_bytes = int(self.lib.rdg_bin_tiles_workspace_bytes(self.n, self.cap, self.H, self.W))
        self.bin_ws = torch.empty(self.bin_bytes, dtype=torch.uint8, device=dev)
        b = RdgBins()
        b.vals_sorted, b.ranges, b.num_rendered = ptr(self.vals), ptr(self.ranges), ptr(self.num_rendered)
        b.region_ids, b.region_masks, b.region_count = ptr(self.region_ids), ptr(self.region_masks), ptr(self.region_count)
        b.region_stride = self.cap
        self.bins = b

    def _write_view(self):
        check(self.lib.rdg_pose_adam(C.byref(self.adam), 0, _lib.stream_ptr()))

    def _forward_bins(self):
        s = _lib.stream_ptr()
        check(self.lib.rdg_preprocess_fwd(C.byref(self.scene), C.byref(self.view_s), C.byref(self.geom_s), s))
        check(self.lib.rdg_bin_tiles(self.n, C.byref(self.geom_s), self.H, self.W, self.cap, C.byref(self.bins), ptr(self.bin_ws),
                                     self.bin_bytes, s))

    def _iteration(self):
        lib, s = self.lib, _lib.stream_ptr()
        self._forward_bins()
        img = _lib.RdgImage()
        img.color, img.depth, img.alpha = ptr(self.color), ptr(self.depth), ptr(self.alpha)
        img.final_T, img.n_contrib = ptr(self.final_T), ptr(self.n_contrib)
        check(lib.rdg_blend_fwd(self.n, C.byref(self.geom_s), C.byref(self.bins), C.byref(self.view_s), C.byref(img), s))
        check(lib.rdg_l2_loss(ptr(self.color), ptr(self.gt), 3, self.H, self.W, ptr(self.step), self.iters, ptr(self.history),
                              ptr(self.dL_dcolor), ptr(self.loss_ws), self.loss_bytes, s))
        self.acc.zero_()
        if engine.config.deterministic:
            check(lib.rdg_blend_bwd_deterministic(self.n, C.byref(self.geom_s), C.byref(self.bins), C.byref(self.view_s),
                                                  C.byref(img), ptr(self.dL_dcolor), None, None, ptr(self.acc),
                                                  ptr(self.det_scratch), self.det_bytes, s))
        else:
            check(lib.rdg_blend_bwd(self.n, C.byref(self.geom_s), C.byref(self.bins), C.byref(self.view_s), C.byref(img),
                                    ptr(self.dL_dcolor), None, None, ptr(self.acc), s))
        check(lib.rdg_preprocess_bwd(C.byref(self.scene), C.byref(self.view_s), C.byref(self.geom_s), ptr(self.acc),
                                     C.byref(self.grads), s))
        check(lib.rdg_pose_adam(C.byref(self.adam), 1, s))

    def _capture(self):
        _lib.set_tunable("deterministic", 1 if engine.config.deterministic else 0)
        self.graph = None
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._iteration()
        self.graph = graph

    def run(self) -> Tuple[torch.Tensor, torch.Tensor]:
        headroom = max(float(engine.config.headroom), 1.0)
        # duplicate capacity: one host read of the count at the initial pose (tile_scan counts past a full buffer)
        self._write_view()
        self._alloc_bins(1)
        self._forward_bins()
        self._alloc_bins(int(int(self.num_rendered[0]) * headroom) + 1)
        # one eager iteration loads every kernel outside the capture; then the pose state starts over
        _lib.set_tunable("deterministic", 1 if engine.config.deterministic else 0)
        self._iteration()
        self.param.copy_(self.pose0)
        for t in (self.exp_avg, self.exp_avg_sq, self.step, self.dV, self.overflow):
            t.zero_()
        self._write_view()
        self._capture()
        done = 0
        while done < self.iters:
            for _ in range(min(CHUNK, self.iters - done)):
                self.graph.replay()
            host = torch.cat([self.step, self.overflow]).cpu()
            done = int(host[0])
            if int(host[1]):
                # a pose saw more tile instances than the buffers hold: nothing was applied at that iteration; grow the
                # buffers from the latched count and continue from the step counter
                self.overflow.zero_()
                self._alloc_bins(int(int(host[2]) * headroom) + 1)
                self._capture()
        return self.vm.view(4, 4).clone(), self.history


def refine_poses(static: Dict[str, torch.Tensor], height: int, width: int, sh_degree: int, bg: torch.Tensor,
                 viewmats: torch.Tensor, projmats: torch.Tensor, tanfovx: Union[float, Sequence[float]],
                 tanfovy: Union[float, Sequence[float]], gts: torch.Tensor, lr: float, iters: int = 1000,
                 ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Refine the pose of V held-out cameras against their ground truth with the static model (the reference's
    PoseOptimizer).  static: raw static-model tensors (dynamic.GaussianParams names, with or without the reference's
    leading '_', e.g. checkpoint.export_models(step)["static"]); bg [3]; viewmats / projmats [V, 4, 4] glm storage; tanfovx /
    tanfovy a float or V floats; gts [V, 3, H, W]; lr the constant Adam learning rate.
    Returns (viewmats_refined [V, 4, 4] glm storage, losses [V, iters]): losses[v, i] is the L2 loss at the pose before
    update i, the refined pose is the one after the last update."""
    V = viewmats.shape[0] if torch.is_tensor(viewmats) and viewmats.dim() == 3 else 0
    if V < 1:
        raise ValueError("refine_poses: viewmats must be a [V, 4, 4] tensor with V >= 1")
    dev = viewmats.device
    if dev.type != "cuda":
        raise ValueError(f"refine_poses: runs on CUDA tensors only, viewmats is on {dev}")
    H, W = int(height), int(width)
    _check("viewmats", viewmats, (V, 4, 4), dev)
    _check("projmats", projmats, (V, 4, 4), dev)
    _check("gts", gts, (V, 3, H, W), dev)
    _check("bg", bg, (3,), dev)
    if not 0 <= int(sh_degree) <= 3:
        raise ValueError(f"refine_poses: sh_degree must be 0..3, got {sh_degree}")
    if int(iters) != iters or iters < 1:
        raise ValueError(f"refine_poses: iters must be an integer >= 1, got {iters}")
    if not lr > 0 or lr == float("inf"):
        raise ValueError(f"refine_poses: lr must be a finite value > 0, got {lr}")
    fovx, fovy = per_view("tanfovx", tanfovx, V), per_view("tanfovy", tanfovy, V)
    st = _static_set(static)
    if st.xyz.device != dev:
        raise ValueError(f"refine_poses: the static model is on {st.xyz.device}, the views on {dev}")
    poses = pose_from_viewmatrix(viewmats)
    out = torch.empty(V, 4, 4, dtype=torch.float32, device=dev)
    losses = torch.empty(V, int(iters), dtype=torch.float32, device=dev)
    for v in range(V):
        view = ViewArgs(height=H, width=W, tanfovx=fovx[v], tanfovy=fovy[v], scale_modifier=1.0, sh_degree=int(sh_degree),
                        viewmatrix=viewmats[v], projmatrix=projmats[v], bg=bg)
        out[v], losses[v] = _PoseLoop(st, view, gts[v], poses[v].contiguous(), float(lr), int(iters)).run()
    return out, losses
