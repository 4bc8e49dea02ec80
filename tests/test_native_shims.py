"""The simple_knn / pytorch3d import shims over the exact grid KNN (rodygs_b200/knn.py, csrc/knn.cu):
RoDyGS's `from simple_knn._C import distCUDA2` and `import pytorch3d.ops as torch3d` resolve from the repo alone.

CPU: the shims import without a GPU and without the oracle, CPU tensors and every unsupported knn_points argument raise.
GPU: distCUDA2 is bit-exact against dist_cuda2_exhaustive below on adversarial clouds; knn_points indices and
distances are bit-exact against rdg_knn and oracle.motion_oracle.knn_points; the gradient of the distances is held
element-wise to a float64 truth; the reference's RigidityLoss computation runs through the shim within the tolerances
of tests/test_gpu_motion.py."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from helpers import elementwise_vs_truth, rel_err
from oracle import motion_oracle as mo

gpu = pytest.mark.gpu


def dist_cuda2_exhaustive(points: torch.Tensor, rows=None, chunk: int = 256) -> torch.Tensor:
    """simple-knn's distCUDA2 (src/model/rodygs_static.py:130-133) by exhaustive search: for each point (or each of
    `rows`) the mean of the squared distances to its 3 nearest OTHER points, ((b0 + b1) + b2) / 3 with b ascending.
    The point itself is excluded by index, not by distance (an exact duplicate is another point at distance 0); the
    distance is (dx*dx + dy*dy) + dz*dz, one rounding per operation in the input precision.  simple-knn is an
    un-vendored submodule absent from the reference snapshot; this restates its recalled contract,
    `(best[0] + best[1] + best[2]) / 3.0f`.  Device-agnostic: every operation rounds the same way on any device."""
    rows = torch.arange(points.shape[0], device=points.device) if rows is None else rows.to(points.device)
    out = torch.empty(rows.shape[0], dtype=points.dtype, device=points.device)
    x, y, z = (c.contiguous() for c in points.detach().unbind(1))
    with torch.no_grad():
        for s in range(0, rows.shape[0], chunk):
            r = rows[s:s + chunk]
            dx, dy, dz = x[r][:, None] - x[None], y[r][:, None] - y[None], z[r][:, None] - z[None]
            d = dx.mul_(dx).add_(dy.mul_(dy)).add_(dz.mul_(dz))          # (dx*dx + dy*dy) + dz*dz
            d[torch.arange(r.shape[0], device=d.device), r] = float("inf")
            b = torch.topk(d, 3, dim=1, largest=False, sorted=True).values
            s3 = (b[:, 0] + b[:, 1]) + b[:, 2]
            # a full tensor, not the scalar 3: torch divides by a scalar as a product with its reciprocal on CUDA
            out[s:s + chunk] = s3 / torch.full_like(s3, 3.0)
    return out


def knn_dist2(query: torch.Tensor, ref: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """Differentiable |query[i] - ref[idx[i, k]]|^2 [n, K] of given neighbours, (dx*dx + dy*dy) + dz*dz in the input
    precision: in float64 the truth for the gradient of knn_points' dists w.r.t. p1 (query) and p2 (ref), which hold
    the same points; in float32 the float32 twin of that truth."""
    nb = ref[idx]
    dx = query[:, None, 0] - nb[..., 0]
    dy = query[:, None, 1] - nb[..., 1]
    dz = query[:, None, 2] - nb[..., 2]
    return (dx * dx + dy * dy) + dz * dz


# ---- CPU ---------------------------------------------------------------------------------------------------------------

def test_shims_import_with_only_the_repo_root_and_no_gpu():
    code = ("import sys\n"
            "from simple_knn._C import distCUDA2\n"
            "import pytorch3d.ops as torch3d\n"
            "torch3d.knn_points; torch3d.knn_gather\n"
            "import simple_knn, pytorch3d\n"
            "assert 'oracle' not in sys.modules\n"
            "print(simple_knn.__file__); print(pytorch3d.__file__)\n")
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    env.update(PYTHONPATH=ROOT, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], cwd="/", env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    for line in out.stdout.split():
        assert os.path.realpath(line).startswith(os.path.realpath(ROOT)), line


def test_shims_never_import_the_oracle():
    for base in ("simple_knn", "pytorch3d"):
        files = [os.path.join(d, f) for d, _, fs in os.walk(os.path.join(ROOT, base)) for f in fs if f.endswith(".py")]
        assert files, base
        for path in files:
            assert not re.search(r"^\s*(from|import)\s+oracle\b", open(path).read(), flags=re.M), path


def test_cpu_tensors_raise():
    from simple_knn._C import distCUDA2
    import pytorch3d.ops as torch3d
    p = torch.rand(64, 3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        distCUDA2(p)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        torch3d.knn_points(p[None], p[None], K=4)


@pytest.mark.parametrize("name", ["lengths1", "lengths2", "norm", "batch", "D", "p2", "K"])
def test_unsupported_knn_points_arguments_raise_naming_them(name):
    import pytorch3d.ops as torch3d
    p = torch.rand(64, 3)
    q = p[None]
    calls = {
        "lengths1": (lambda: torch3d.knn_points(q, q, lengths1=torch.tensor([64]), K=4), "lengths1"),
        "lengths2": (lambda: torch3d.knn_points(q, q, lengths2=torch.tensor([64]), K=4), "lengths2"),
        "norm": (lambda: torch3d.knn_points(q, q, norm=1, K=4), "norm=1"),
        "batch": (lambda: torch3d.knn_points(torch.rand(2, 64, 3), torch.rand(2, 64, 3), K=4), r"p1.*batch"),
        "D": (lambda: torch3d.knn_points(torch.rand(1, 64, 2), torch.rand(1, 64, 2), K=4), "D=2"),
        "p2": (lambda: torch3d.knn_points(q, p.clone()[None], K=4), "p2"),
        "K": (lambda: torch3d.knn_points(q, q, K=17), "K=17"),
    }
    fn, pattern = calls[name]
    with pytest.raises(NotImplementedError, match=pattern):
        fn()


def test_knn_gather_indexes_and_refuses_lengths():
    import pytorch3d.ops as torch3d
    x = torch.rand(1, 50, 5)
    idx = torch.randint(0, 50, (1, 20, 4))
    assert torch.equal(torch3d.knn_gather(x, idx), x[0][idx[0]][None])
    with pytest.raises(NotImplementedError, match="lengths"):
        torch3d.knn_gather(x, idx, lengths=torch.tensor([50]))


def test_native_argument_errors_without_a_gpu():
    from rodygs_b200 import _lib
    lib = _lib.load()
    one = (ctypes.c_float * 16)()
    assert lib.rdg_knn3_mean_dist2(3, one, one, one, 1 << 20, None) == -1
    assert b"at least 4" in lib.rdg_last_error()
    assert lib.rdg_knn3_mean_dist2(8, None, one, one, 1 << 20, None) == -1
    assert lib.rdg_knn_dist2_bwd(8, 3, None, one, one, one, None, None) == -1
    assert lib.rdg_knn_dist2_bwd(8, 17, one, one, one, one, None, None) == -1


def test_exhaustive_dist_cuda2_known_answer():
    """The exhaustive reference against a plain float32 loop: 3 smallest over j != i, ((b0 + b1) + b2) / 3."""
    gen = torch.Generator().manual_seed(0)
    p = torch.rand(200, 3, generator=gen)
    p[150] = p[10]                   # a pair; for row 150 the duplicate has the lower index
    p[50:55] = torch.tensor([2.0, 2.0, 2.0])   # a 5-fold stack: 4 others at distance 0
    pn = p.numpy()
    ref = []
    for i in range(len(pn)):
        d = []
        for j in range(len(pn)):
            if j != i:
                dx, dy, dz = pn[i] - pn[j]                  # numpy float32 scalars: one rounding per operation
                d.append((dx * dx + dy * dy) + dz * dz)
        d.sort()
        ref.append(((d[0] + d[1]) + d[2]) / np.float32(3))
    got = dist_cuda2_exhaustive(p, chunk=64)
    assert torch.equal(got, torch.tensor(np.array(ref)))
    assert (got[50:55] == 0).all() and got[10] == got[150] and got[10] > 0
    assert torch.equal(dist_cuda2_exhaustive(p, rows=torch.tensor([150, 3, 52])), got[[150, 3, 52]])


# ---- GPU: distCUDA2 ----------------------------------------------------------------------------------------------------

def _dist_clouds():
    gen = torch.Generator().manual_seed(5)
    cube = torch.rand(50_000, 3, generator=gen) * 4 - 2
    centres = torch.randn(8, 3, generator=gen) * 2
    blobs = centres[torch.randint(0, 8, (20_000,), generator=gen)] + torch.randn(20_000, 3, generator=gen) * 0.05
    blobs[::1000] = torch.randn(20, 3, generator=gen) * 200            # far outliers
    # MASt3R-like: points on a floor and two walls, so the volume-sized grid crowds the cells they cross
    m = 60_000
    uv = torch.rand(m, 2, generator=gen) * 3
    which = torch.randint(0, 3, (m,), generator=gen)
    surface = torch.zeros(m, 3)
    surface[which == 0] = torch.stack([uv[:, 0], uv[:, 1], torch.zeros(m)], 1)[which == 0]
    surface[which == 1] = torch.stack([torch.zeros(m), uv[:, 0], uv[:, 1]], 1)[which == 1]
    surface[which == 2] = torch.stack([uv[:, 0], torch.zeros(m), uv[:, 1]], 1)[which == 2]
    flat = torch.rand(20_000, 3, generator=gen)
    flat[:, 2] = 0.5
    dup = torch.rand(8_000, 3, generator=gen)
    dup[3000:3500] = dup[:500]                     # pairs; rows 3000.. have their duplicate at a LOWER index
    dup[7000:7005] = torch.tensor([1.5, 1.5, 1.5])  # a 5-fold stack: mean 0
    four = torch.rand(4, 3, generator=gen)
    return {"cube50k": cube, "blobs_outliers": blobs, "surface": surface, "flat": flat, "duplicates": dup, "n4": four}


@gpu
@pytest.mark.parametrize("name", ["cube50k", "blobs_outliers", "surface", "flat", "duplicates", "n4"])
def test_dist_cuda2_bit_exact(name):
    from simple_knn._C import distCUDA2
    p = _dist_clouds()[name].cuda()
    got = distCUDA2(p)
    ref = dist_cuda2_exhaustive(p)                  # on the device (test_exhaustive_dist_cuda2_is_device_agnostic)
    assert got.dtype == torch.float32 and got.shape == (p.shape[0],)
    assert torch.equal(got, ref), (name, (got - ref).abs().max().item())
    if name == "duplicates":
        assert (got[7000:7005] == 0).all()
        assert torch.equal(got[3000:3500], got[:500])


@gpu
def test_exhaustive_dist_cuda2_is_device_agnostic():
    p = _dist_clouds()["duplicates"][:3000]
    assert torch.equal(dist_cuda2_exhaustive(p).cuda(), dist_cuda2_exhaustive(p.cuda()))


@gpu
def test_dist_cuda2_non_contiguous_input():
    from simple_knn._C import distCUDA2
    base = torch.rand(3, 30_000, generator=torch.Generator().manual_seed(9)).cuda()
    p = base.t()
    assert not p.is_contiguous()
    assert torch.equal(distCUDA2(p), dist_cuda2_exhaustive(p.contiguous()))


@gpu
def test_dist_cuda2_2m_points_against_exhaustive_rows():
    from simple_knn._C import distCUDA2
    gen = torch.Generator().manual_seed(13)
    n = 2_000_000
    p = (torch.rand(n, 3, generator=gen) * torch.tensor([8.0, 4.0, 2.0])).cuda()
    rows = torch.randint(0, n, (4096,), generator=gen).cuda()
    got = distCUDA2(p)
    assert torch.equal(got[rows], dist_cuda2_exhaustive(p, rows=rows))


@gpu
def test_dist_cuda2_rejects_bad_input():
    from simple_knn._C import distCUDA2
    with pytest.raises(RuntimeError, match="at least 4"):
        distCUDA2(torch.rand(3, 3).cuda())
    with pytest.raises(RuntimeError, match="dtype"):
        distCUDA2(torch.rand(10, 3, dtype=torch.float64).cuda())
    with pytest.raises(RuntimeError, match=r"\[P, 3\]"):
        distCUDA2(torch.rand(10, 2).cuda())


# ---- GPU: knn_points ---------------------------------------------------------------------------------------------------

def _knn_cloud():
    gen = torch.Generator().manual_seed(17)
    p = torch.rand(4000, 3, generator=gen)
    p[2000:2300] = p[:300]                          # pairs at distance 0, the lower index first
    p[3990:3995] = torch.tensor([1.2, 1.2, 1.2])    # a 5-fold stack
    return p


@gpu
@pytest.mark.parametrize("K", [1, 3, 8, 16])
def test_knn_points_bit_exact(K):
    import pytorch3d.ops as torch3d
    from rodygs_b200 import motion_reg as mr
    p = _knn_cloud()
    pc = p.cuda()
    dists, idx, knn = torch3d.knn_points(pc[None], pc[None], K=K)
    assert knn is None and idx.dtype == torch.int64 and dists.shape == idx.shape == (1, p.shape[0], K)
    d_ref, i_ref = mo.knn_points(p, K)
    _, i_native = mr.knn_points(pc, K)
    assert torch.equal(idx[0].cpu(), i_ref)
    assert torch.equal(idx[0], i_native.long())
    assert torch.equal(dists[0].cpu(), d_ref)
    # return_sorted=False still returns the sorted result; version is ignored
    d2, i2, nn = torch3d.knn_points(pc[None], pc[None], K=K, version=0, return_nn=True, return_sorted=False)
    assert torch.equal(i2, idx) and torch.equal(d2, dists)
    assert torch.equal(nn[0], pc[idx[0]])
    assert torch.equal(torch3d.knn_gather(pc[None], idx)[0], pc[idx[0]])


@gpu
@pytest.mark.parametrize("which", ["both", "p1", "p2"])
def test_knn_points_distance_gradient_against_float64(which):
    """d/dp of (dists * w).sum(), element-wise against float64 autograd of the same neighbour distances;
    `which` says which of p1 / p2 requires grad (both from one leaf, or only one side)."""
    import pytorch3d.ops as torch3d
    K = 8
    p = _knn_cloud()
    w = torch.randn(1, p.shape[0], K, generator=torch.Generator().manual_seed(23))
    leaf = p.cuda().requires_grad_(True)
    p1 = leaf[None] if which in ("both", "p1") else leaf.detach()[None]
    p2 = leaf[None] if which in ("both", "p2") else leaf.detach()[None]
    dists, idx, _ = torch3d.knn_points(p1, p2, K=K)
    (got,) = torch.autograd.grad((dists * w.cuda()).sum(), leaf)
    idx = idx[0].cpu()
    refs = []
    for dt in (torch.float32, torch.float64):
        lv = p.to(dt).requires_grad_(True)
        q = lv if which in ("both", "p1") else lv.detach()
        r = lv if which in ("both", "p2") else lv.detach()
        (gr,) = torch.autograd.grad((knn_dist2(q, r, idx) * w[0].to(dt)).sum(), lv)
        refs.append(gr)
    ok, r_cu, r_32 = elementwise_vs_truth(got, refs[0], refs[1])
    assert ok, (which, r_cu, r_32)


@gpu
@pytest.mark.parametrize("tag,mode", [("rigid_cfg", ("distance_preserving", "surface")), ("rigid_surface", ("surface",)),
                                      ("rigid_dp", ("distance_preserving",)), ("rigid_coeff", ("coeff",))])
def test_reference_rigidity_through_the_shim(monkeypatch, tag, mode):
    """oracle.motion_oracle.rigidity is the reference's RigidityLoss.forward; its neighbour search is swapped for the
    drop-in knn_points (forward and backward on the GPU), and the result must still match the reference's golden."""
    import pytorch3d.ops as torch3d
    from test_oracle_motion import load_motion

    def shim_knn(points, K):
        pc = points.cuda()
        dists, idx, _ = torch3d.knn_points(pc[None], pc[None], K=K)
        return dists[0].cpu(), idx[0].cpu()

    monkeypatch.setattr(mo, "knn_points", shim_knn)
    g = load_motion()
    lv = {k: g[k].clone().requires_grad_(True) for k in ("xyz", "coeff", "table", "pred_tr")}
    loss, _ = mo.rigidity(lv["xyz"], lv["coeff"], g["fdc"], lv["pred_tr"], lv["table"], g[f"{tag}/indice"],
                          g.get(f"{tag}/time_indices"), K=int(g["K"]), mode=mode)
    ref = g[f"{tag}/loss"].item()
    assert abs(loss.item() - ref) <= 1e-5 * max(1.0, abs(ref)), (tag, loss.item(), ref)
    grads = torch.autograd.grad(loss, list(lv.values()), allow_unused=True)
    for k, gr in zip(lv, grads):
        key = f"{tag}/d_{k}"
        if key not in g:
            assert gr is None or gr.abs().max().item() == 0, (tag, k)
            continue
        assert rel_err(gr, g[key]) < 1e-3, (tag, k, rel_err(gr, g[key]))
