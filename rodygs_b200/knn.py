"""The exact grid KNN of csrc/knn.cu behind the two third-party KNN calls RoDyGS makes:

    simple_knn._C.distCUDA2(points)                     src/model/rodygs_static.py:17, :130-133 (initial scales)
    pytorch3d.ops.knn_points(p[None], p[None], K)       src/trainer/losses.py:18, :238-239 (RigidityLoss)

Neither upstream source is in the reference snapshot (simple-knn and pytorch3d are un-vendored), so the signatures and
semantics here are recalled from upstream and unpinned, like diff_gauss_pose: distCUDA2 is the mean squared distance to
the 3 nearest OTHER points, (best[0] + best[1] + best[2]) / 3.0f; knn_points returns squared distances with gradients.
The import shims simple_knn/ and pytorch3d/ re-export these.  There is no CPU path: CPU tensors raise.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import check, ptr
from .motion_reg import _ws, knn_points


def _points(t: torch.Tensor, what: str) -> torch.Tensor:
    _lib.require_cuda(t)
    if t.dtype != torch.float32:
        raise RuntimeError(f"{what}: float32 points expected, got {t.dtype}")
    if t.dim() != 2 or t.shape[1] != 3:
        raise RuntimeError(f"{what}: points of shape [P, 3] expected, got {list(t.shape)}")
    return t.detach().contiguous()


def dist_cuda2(points: torch.Tensor) -> torch.Tensor:
    """simple-knn's distCUDA2: [P, 3] float32 CUDA -> [P] float32, the mean squared distance from each point to its 3
    nearest other points (the point itself is excluded by index, so an exact duplicate counts at distance 0).  No
    autograd.  P >= 4."""
    lib = _lib.load()
    p = _points(points, "distCUDA2")
    n = p.shape[0]
    out = torch.empty(n, dtype=torch.float32, device=p.device)
    nbytes = int(lib.rdg_knn_workspace_bytes(n))
    ws = _ws(nbytes, p.device)
    check(lib.rdg_knn3_mean_dist2(n, ptr(p), ptr(out), ptr(ws), nbytes, _lib.stream_ptr()))
    return out


class KnnSelfFn(torch.autograd.Function):
    """(query, ref, K) -> (dist2 [P, K], idx [P, K] int32): the K nearest of the P points of one cloud for each of its
    points, itself included.  `query` and `ref` hold the same points (pytorch3d's p1 and p2); they are separate inputs
    so that each gets only its own part of the gradient, whichever of them requires grad."""

    @staticmethod
    def forward(ctx, query, ref, K):
        p = _points(query, "knn_points")
        d2, idx = knn_points(p, K)
        ctx.save_for_backward(p, idx)
        ctx.mark_non_differentiable(idx)
        return d2, idx

    @staticmethod
    def backward(ctx, g, _gidx):
        p, idx = ctx.saved_tensors
        n, K = idx.shape
        d_query = torch.empty_like(p) if ctx.needs_input_grad[0] else None
        d_ref = torch.zeros_like(p) if ctx.needs_input_grad[1] else None
        g = g.detach().float().contiguous()
        check(_lib.load().rdg_knn_dist2_bwd(n, K, ptr(p), ptr(idx), ptr(g), ptr(d_query), ptr(d_ref), _lib.stream_ptr()))
        return d_query, d_ref, None
