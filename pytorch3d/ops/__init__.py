"""pytorch3d.ops.knn_points / knn_gather for the one call RoDyGS makes, `knn_points(p[None], p[None], K=K)`
(src/trainer/losses.py:238-239), on the exact grid KNN of rodygs_b200 (csrc/knn.cu).

This is a partial pytorch3d that shadows a real one on PYTHONPATH (see pytorch3d/__init__.py).  The signatures and
return types are recalled from upstream pytorch3d, whose source is not in the reference snapshot, so they are unpinned
like diff_gauss_pose.  What is built: batch 1, D = 3, p1 and p2 views of the same points (same storage, shape and
strides), norm=2 (squared Euclidean distances).  Results are always sorted ascending, with exact ties towards the lower
index, so `return_sorted=False` also returns them sorted; `version` is ignored.  Two different clouds, batch > 1,
`lengths1` / `lengths2`, `norm=1`, D != 3 and K > 16 raise NotImplementedError.
"""
from collections import namedtuple

import torch

from rodygs_b200.knn import KnnSelfFn

_KNN = namedtuple("KNN", "dists idx knn")

__all__ = ["knn_points", "knn_gather"]


def _unsupported(arg: str, why: str):
    raise NotImplementedError(f"knn_points: {arg} is not supported here ({why}); only knn_points(p[None], p[None], K) "
                              "of one cloud is built")


def knn_points(p1: torch.Tensor, p2: torch.Tensor, lengths1=None, lengths2=None, norm: int = 2, K: int = 1,
               version: int = -1, return_nn: bool = False, return_sorted: bool = True):
    """p1 = p2 = p[None] ([1, P, 3] float32 CUDA) -> KNN(dists [1, P, K] squared distances ascending, differentiable
    w.r.t. p1 and p2; idx [1, P, K] int64, each point's own index first unless an exact duplicate has a lower index;
    knn = p2 gathered at idx [1, P, K, 3] if return_nn, else None)."""
    if lengths1 is not None:
        _unsupported("lengths1", "ragged batches")
    if lengths2 is not None:
        _unsupported("lengths2", "ragged batches")
    if norm != 2:
        _unsupported(f"norm={norm}", "only norm=2, squared Euclidean distances")
    if p1.dim() != 3 or p1.shape[0] != 1:
        _unsupported(f"p1 of shape {list(p1.shape)}", "batch > 1; p1 must be [1, P, 3]")
    if p1.shape[2] != 3:
        _unsupported(f"D={p1.shape[2]}", "only 3-D points")
    if not (p2.device == p1.device and p2.data_ptr() == p1.data_ptr() and p2.shape == p1.shape
            and p2.stride() == p1.stride()):
        _unsupported("p2", "two different clouds; p2 must be a view of the same points as p1")
    if not 1 <= K <= 16:
        _unsupported(f"K={K}", "K must be in 1..16")
    dists, idx = KnnSelfFn.apply(p1[0], p2[0], int(K))
    idx = idx.long()[None]
    return _KNN(dists[None], idx, knn_gather(p2, idx) if return_nn else None)


def knn_gather(x: torch.Tensor, idx: torch.Tensor, lengths=None) -> torch.Tensor:
    """x [N, P2, C], idx [N, P1, K] -> x gathered at idx, [N, P1, K, C] (plain indexing, differentiable w.r.t. x)."""
    if lengths is not None:
        raise NotImplementedError("knn_gather: lengths is not supported here (ragged batches)")
    return x[torch.arange(x.shape[0], device=x.device)[:, None, None], idx]
