"""Export as a 3D Gaussian Splatting PLY file, CPU side: rdg_export_3dgs's argument refusals, SplatTrainStep.export_3dgs's host
checks, the kernel's compile report, rodygs_b200.ply's writer and reader, and the float64 twin of a dynamic record held to
closed forms (the twin is the yardstick of the GPU tests in test_gpu_export.py)."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from test_checkpoint import _cpu_step

FLT_MIN = float(np.finfo(np.float32).tiny)


# ============================================================ the twin ==

def rot64(q):
    """rdg_project's R(q) [..., 3, 3] in float64 from q [..., 4] = (r, x, y, z) as it is (not normalised)"""
    r, x, y, z = q.double().unbind(-1)
    return torch.stack([torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y)], -1),
                        torch.stack([2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x)], -1),
                        torch.stack([2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], -1)], -2)


def quat_of(U):
    """unit quaternion (w, x, y, z), w >= 0, of rotation matrices U [n, 3, 3] (float64)"""
    m = U
    cand = torch.stack([1 + m[:, 0, 0] + m[:, 1, 1] + m[:, 2, 2], 1 + m[:, 0, 0] - m[:, 1, 1] - m[:, 2, 2],
                        1 - m[:, 0, 0] + m[:, 1, 1] - m[:, 2, 2], 1 - m[:, 0, 0] - m[:, 1, 1] + m[:, 2, 2]], 1)
    k = cand.argmax(1)
    f = 2 * cand.gather(1, k[:, None])[:, 0].clamp(min=0).sqrt()
    a, b, c = m[:, 2, 1] - m[:, 1, 2], m[:, 0, 2] - m[:, 2, 0], m[:, 1, 0] - m[:, 0, 1]
    d, e, g = m[:, 0, 1] + m[:, 1, 0], m[:, 0, 2] + m[:, 2, 0], m[:, 1, 2] + m[:, 2, 1]
    q = torch.stack([torch.stack([f / 4, a / f, b / f, c / f], 1), torch.stack([a / f, f / 4, d / f, e / f], 1),
                     torch.stack([b / f, d / f, f / 4, g / f], 1), torch.stack([c / f, e / f, g / f, f / 4], 1)], 1)
    q = q[torch.arange(U.shape[0]), k]
    q = q / q.norm(dim=1, keepdim=True)
    return torch.where(q[:, :1] < 0, -q, q)


def twin(qp, s):
    """float64 twin of the dynamic record from the float32 q' [n, 4] and s = exp(scaling) [n, 3]: (Sigma [n, 3, 3],
    rot [n, 4], scale [n, 3]).  Sigma = M M^T, M = R(q') diag(s); Sigma = U diag(lambda) U^T with det U = +1; rot = the
    quaternion of U with rot_0 >= 0; scale = 0.5 log(max(lambda, FLT_MIN))."""
    M = rot64(qp) * s.double()[:, None, :]
    sigma = M @ M.transpose(1, 2)
    lam, U = torch.linalg.eigh(sigma)
    U = U.clone()
    U[:, :, 0] *= torch.linalg.det(U).sign()[:, None]
    return sigma, quat_of(U), 0.5 * lam.clamp(min=FLT_MIN).log()


def sigma_of(rot, scale):
    """R(rot / |rot|) diag(exp(2 scale)) R^T in float64: the covariance a viewer draws from a record's rot and scale"""
    q = rot.double() / rot.double().norm(dim=1, keepdim=True)
    R = rot64(q)
    return R @ torch.diag_embed(torch.exp(2 * scale.double())) @ R.transpose(1, 2)


def _rel(a, b):
    return ((a - b).flatten(1).norm(dim=1) / b.flatten(1).norm(dim=1)).max().item()


def _quarter_turn_z():
    return torch.tensor([[np.cos(np.pi / 4), 0.0, 0.0, np.sin(np.pi / 4)]], dtype=torch.float64)


def test_twin_unit_quaternion():
    """|q'| = 1: R(q') is a rotation, Sigma = R diag(s^2) R^T, and (rot, scale) is R and log s up to the axes' order."""
    g = torch.Generator().manual_seed(0)
    q = torch.randn(64, 4, generator=g, dtype=torch.float64)
    q = q / q.norm(dim=1, keepdim=True)
    s = torch.exp(torch.randn(64, 3, generator=g, dtype=torch.float64))
    R = rot64(q)
    closed = R @ torch.diag_embed(s * s) @ R.transpose(1, 2)
    sigma, rot, scale = twin(q, s)
    assert _rel(sigma, closed) < 1e-13
    assert _rel(sigma_of(rot, scale), closed) < 1e-12
    assert ((rot.norm(dim=1) - 1).abs() < 1e-14).all() and (rot[:, 0] >= 0).all()
    assert torch.allclose(scale.sort(1).values, s.log().sort(1).values, rtol=0, atol=1e-12)


def test_twin_isotropic_scale():
    """s_0 = s_1 = s_2: Sigma = s^2 R(q') R(q')^T for any q', unit or not."""
    g = torch.Generator().manual_seed(1)
    q = torch.randn(64, 4, generator=g, dtype=torch.float64) * 0.6
    s = torch.exp(torch.randn(64, 1, generator=g, dtype=torch.float64)).expand(64, 3)
    R = rot64(q)
    closed = (s[:, 0] ** 2)[:, None, None] * (R @ R.transpose(1, 2))
    sigma, rot, scale = twin(q, s)
    assert _rel(sigma, closed) < 1e-13
    assert _rel(sigma_of(rot, scale), closed) < 1e-12


def test_twin_quaternion_longer_than_one():
    """q' = lambda q^ with lambda^2 = 1.1 and q^ a quarter turn about z: R(q') = (1 - lambda^2) I + lambda^2 R(q^), and for
    isotropic s the covariance is s^2 diag(1.22, 1.22, 1) - two axes sqrt(1.22) = 1.105 times longer than a viewer draws
    from the normalised q'.  With anisotropic s the exported Sigma differs from that naive export by more than 1 %."""
    lam = np.sqrt(1.1)
    qp = lam * _quarter_turn_z()
    s = torch.tensor([[0.3, 0.3, 0.3]], dtype=torch.float64)
    sigma, rot, scale = twin(qp, s)
    closed = 0.09 * torch.diag(torch.tensor([1.22, 1.22, 1.0], dtype=torch.float64))[None]
    assert _rel(sigma, closed) < 1e-14
    assert _rel(sigma_of(rot, scale), closed) < 1e-12
    assert torch.allclose(scale.sort(1).values, torch.tensor([[np.log(0.3), 0.5 * np.log(0.09 * 1.22),
                                                               0.5 * np.log(0.09 * 1.22)]], dtype=torch.float64), atol=1e-12)
    s = torch.tensor([[0.5, 0.2, 0.05]], dtype=torch.float64)
    sigma = twin(qp, s)[0]
    Rq = torch.tensor([[[1 - 1.1, -1.1, 0], [1.1, 1 - 1.1, 0], [0, 0, 1]]], dtype=torch.float64)
    assert _rel(sigma, Rq @ torch.diag_embed(s * s) @ Rq.transpose(1, 2)) < 1e-14
    naive = sigma_of(qp / qp.norm(), s.log())
    assert _rel(naive, sigma) > 0.01


def test_twin_singular_covariance():
    """q' = lambda q^ with lambda^2 = 0.5 and q^ a half turn about z: R(q') = diag(0, 0, 1), Sigma = diag(0, 0, s_2^2) is
    singular.  The record stays finite and rebuilds Sigma to 1e-16 absolute.  An exact zero eigenvalue (here a zero scale)
    meets the FLT_MIN floor: scale = 0.5 log FLT_MIN."""
    qp = np.sqrt(0.5) * torch.tensor([[0.0, 0.0, 0.0, 1.0]], dtype=torch.float64)
    s = torch.tensor([[0.4, 0.7, 0.25]], dtype=torch.float64)
    sigma, rot, scale = twin(qp, s)
    closed = torch.diag(torch.tensor([0.0, 0.0, 0.0625], dtype=torch.float64))[None]
    assert (sigma - closed).abs().max() < 1e-16
    assert torch.isfinite(rot).all() and torch.isfinite(scale).all()
    assert (scale.sort(1).values[0, :2] < 0.5 * np.log(1e-30)).all()     # two axes of no extent
    assert (sigma_of(rot, scale) - closed).abs().max() < 1e-16
    sigma, rot, scale = twin(_quarter_turn_z(), torch.tensor([[0.0, 0.7, 0.25]], dtype=torch.float64))
    assert torch.isfinite(rot).all() and scale.min().item() == 0.5 * np.log(FLT_MIN)
    assert (sigma_of(rot, scale) - sigma).abs().max() < 1e-16


# ============================================================ the ABI ==

def test_abi_refuses_bad_arguments_without_a_gpu():
    from rodygs_b200 import _lib
    lib = _lib.load()
    buf = (C.c_float * 64)()
    a = C.addressof(buf)
    scene = _lib.RdgScene()
    scene.n_static, scene.raw = 4, 1

    def export(sc=scene, deg=3, rec=a):
        return lib.rdg_export_3dgs(None if sc is None else C.byref(sc), deg, rec, None)

    def refused(msg, **kw):
        return export(**kw) == -1 and msg.encode() in lib.rdg_last_error()

    assert refused("null argument", sc=None)
    scene.n_static = -1
    assert refused("negative count")
    scene.n_static, scene.raw = 4, 0
    assert refused("raw must be 1")
    scene.raw, scene.colors_precomp = 1, a
    assert refused("colors_precomp must be NULL")
    scene.colors_precomp = None
    for deg in (-1, 4):
        assert refused("sh_degree must be 0..3", deg=deg)
    assert refused("null argument", rec=None)
    assert refused("8-byte aligned", rec=a + 4)
    assert refused("null static parameter")
    st = scene.st
    st.xyz = st.scaling = st.rotation = st.opacity = st.sh_dc = a
    assert refused("null static parameter")                                   # sh_rest missing at degree 3
    st.sh_rest, st.sh_dc_stride, st.sh_rest_stride = a, 3, 44
    assert refused("SH stride")
    st.sh_rest_stride, st.sh_dc_stride = 45, 2
    assert refused("SH stride")
    st.sh_dc_stride = 3
    scene.n_dynamic, scene.use_deform, scene.num_basis, scene.num_times = 4, 1, 16, 5
    assert refused("null dynamic parameter")
    dy = scene.dy
    dy.xyz = dy.scaling = dy.rotation = dy.opacity = dy.sh_dc = dy.sh_rest = a
    dy.sh_dc_stride, dy.sh_rest_stride = 3, 45
    for nb in (0, 17):
        scene.num_basis = nb
        assert refused("num_basis out of range")
    scene.num_basis, scene.num_times = 16, 0
    assert refused("num_times out of range")
    scene.num_times = 5
    scene.motion_coeff = scene.time_ind = scene.table = a
    assert refused("null deformation input")                                  # basis_t missing
    scene.basis_t, scene.table = a, None
    assert refused("null deformation input")
    scene.n_static = scene.n_dynamic = 0
    assert export(rec=None) == 0                                               # nothing to do: no launch


def test_export_checks_its_arguments_on_the_host():
    step = _cpu_step(n=50)
    bt = torch.zeros(16, 7)
    for bad in (None, bt[:8], bt.double(), torch.zeros(7, 16).t(), torch.zeros(16, 7, 1)):
        with pytest.raises(ValueError, match="basis_t must be a contiguous float32 tensor of shape \\(16, 7\\)"):
            step.export_3dgs(bad)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):        # no CPU fallback
        step.export_3dgs(bt)


def test_export_kernel_does_not_spill():
    """`-Xptxas -v` of export.cu (its own -fmad=false flags): no spills and no stack frame."""
    from rodygs_b200 import build
    with tempfile.TemporaryDirectory() as tmp:
        r = subprocess.run([build._nvcc(), *build.ARCH, *build.COMMON, *build.SOURCES["export.cu"], "-Xptxas", "-v", "-c",
                            os.path.join(build.CSRC, "export.cu"), "-o", os.path.join(tmp, "export.o")],
                           capture_output=True, text=True, check=True)
    assert build.SOURCES["export.cu"] == ["-fmad=false"]
    info, name = {}, None
    for line in r.stderr.splitlines():
        hit = re.search(r"Compiling entry function '(\w+)'", line)
        if hit:
            name = hit.group(1)
        elif name and "spill" in line:
            info[name] = line.strip()
    assert len(info) == 1 and "export_3dgs_kernel" in next(iter(info)), sorted(info)
    for n, line in info.items():
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in line, (n, line)


# ============================================================ the file ==

def _3dgs_attributes():
    """GaussianModel.construct_list_of_attributes of 3DGS, restated for features_dc [n,3,1] and features_rest [n,3,15]"""
    names = ["x", "y", "z", "nx", "ny", "nz"]
    names += [f"f_dc_{i}" for i in range(1 * 3)]
    names += [f"f_rest_{i}" for i in range(15 * 3)]
    names.append("opacity")
    names += [f"scale_{i}" for i in range(3)]
    names += [f"rot_{i}" for i in range(4)]
    return names


def _records(n, seed=0):
    """random records in the exported layout (normals 0), with a few special values"""
    g = torch.Generator().manual_seed(seed)
    r = torch.randn(n, 62, generator=g)
    r[:, 3:6] = 0.0
    if n > 3:
        r[0, 0], r[1, 60], r[2, 10], r[3, 55] = float("inf"), -0.0, 1e-42, -3.4e38
    return r


def _as_records(d):
    """the static model of read_ply's dict back as [n, 62] records"""
    st = d["static"]
    n = st["_xyz"].shape[0]
    return torch.cat([st["_xyz"], torch.zeros(n, 3), st["_features_dc"].reshape(n, 3),
                      st["_features_rest"].transpose(1, 2).reshape(n, 45), st["_opacity"], st["_scaling"],
                      st["_rotation"]], 1)


def test_header_is_the_3dgs_layout_and_the_size_is_248_bytes_a_gaussian():
    from rodygs_b200 import ply
    assert ply.PLY_PROPERTIES == _3dgs_attributes() and ply.RECORD_FLOATS == 62
    want = ("ply\nformat binary_little_endian 1.0\nelement vertex 7\n"
            + "".join(f"property float {n}\n" for n in _3dgs_attributes()) + "end_header\n")
    assert ply.ply_header(7) == want.encode("ascii")
    with tempfile.TemporaryDirectory() as tmp:
        for n in (0, 1, 7, 1000):
            path = os.path.join(tmp, f"s{n}.ply")
            ply.write_ply(path, _records(n))
            assert os.path.getsize(path) == len(ply.ply_header(n)) + 248 * n
            with open(path, "rb") as f:
                assert f.read(len(ply.ply_header(n))) == ply.ply_header(n)


def test_round_trip_is_bit_exact():
    from rodygs_b200 import checkpoint, ply
    with tempfile.TemporaryDirectory() as tmp:
        for n in (0, 1, 300):
            rec = _records(n, seed=n)
            path = os.path.join(tmp, "s.ply")
            ply.write_ply(path, rec)
            d = ply.read_ply(path)
            assert torch.equal(_as_records(d).view(torch.int32), rec.view(torch.int32)), n
            ply.write_ply(path, rec.numpy())                                   # numpy in, same bytes
            assert torch.equal(_as_records(ply.read_ply(path)).view(torch.int32), rec.view(torch.int32))
            assert d["dynamic"]["_xyz"].shape == (0, 3) and d["dynamic"]["_motion_coeff"].shape == (0, 1, 16)
            assert torch.equal(d["motion"]["table"], torch.zeros(1, 16, 7)) and d["motion"]["spatial_lr_scale"] == 1.0
            scene = checkpoint.import_models(d)                                # a scene SplatTrainStep takes
            assert scene["static"]["features_rest"].shape == (n, 15, 3) and scene["time_ind"].shape == (0,)
            assert torch.equal(scene["static"]["rotation"], rec[:, 58:62])
        with pytest.raises(ValueError, match="float32 array of shape \\[N, 62\\]"):
            ply.write_ply(path, torch.zeros(3, 61))
        with pytest.raises(ValueError, match="must be float32"):
            ply.write_ply(path, torch.zeros(3, 62, dtype=torch.float64))


def _write_custom(path, names, rows, fmt="binary_little_endian", types=None, first="vertex", body=None, n=None):
    n = rows.shape[0] if n is None else n
    types = types or ["float"] * len(names)
    head = ["ply", f"format {fmt} 1.0", "comment written by a test", f"element {first} {n}"]
    head += [f"property {t} {nm}" for t, nm in zip(types, names)] + ["end_header"]
    with open(path, "wb") as f:
        f.write(("\n".join(head) + "\n").encode())
        f.write(np.ascontiguousarray(rows, dtype="<f4").tobytes() if body is None else body)


@pytest.mark.parametrize("degree", [0, 1, 2])
def test_lower_degree_files_fill_the_missing_coefficients_with_zero(degree):
    """A degree-d file has 3 ((d + 1)^2 - 1) f_rest properties, channel-major (f_rest_{c R + j}); the reader puts them in
    the first coefficients and zeros the others.  Extra properties (here an 'extra' column and normals) are ignored, and
    properties are found by name, not by position."""
    from rodygs_b200 import ply
    R = (degree + 1) ** 2 - 1
    names = ["extra", "rot_0", "rot_1", "rot_2", "rot_3", "x", "y", "z", "nx", "ny", "nz", "f_dc_0", "f_dc_1", "f_dc_2"]
    names += [f"f_rest_{i}" for i in range(3 * R)] + ["opacity", "scale_0", "scale_1", "scale_2"]
    g = torch.Generator().manual_seed(degree)
    rows = torch.randn(37, len(names), generator=g).numpy()
    col = {nm: i for i, nm in enumerate(names)}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "d.ply")
        _write_custom(path, names, rows)
        st = ply.read_ply(path)["static"]
    assert np.array_equal(st["_rotation"].numpy(), rows[:, [col[f"rot_{i}"] for i in range(4)]])
    assert np.array_equal(st["_xyz"].numpy(), rows[:, [col["x"], col["y"], col["z"]]])
    assert np.array_equal(st["_opacity"].numpy()[:, 0], rows[:, col["opacity"]])
    rest = st["_features_rest"].numpy()
    for c in range(3):
        for j in range(15):
            want = rows[:, col[f"f_rest_{c * R + j}"]] if j < R else 0.0
            assert np.array_equal(rest[:, j, c], np.broadcast_to(want, (37,))), (c, j)


def test_reader_refusals():
    from rodygs_b200 import ply
    names = ply.PLY_PROPERTIES
    rows = _records(5).numpy()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "bad.ply")

        def refused(match, **kw):
            _write_custom(path, kw.pop("names", names), kw.pop("rows", rows), **kw)
            with pytest.raises(ValueError, match=match):
                ply.read_ply(path)

        refused("is 'ascii 1.0'; only binary_little_endian", fmt="ascii")
        refused("is 'binary_big_endian 1.0'; only binary_little_endian", fmt="binary_big_endian")
        refused("vertex property 'double x' is not float", types=["double"] + ["float"] * 61)
        refused("vertex property 'uchar red' is not float", names=names + ["red"], rows=np.zeros((5, 63), np.float32),
                types=["float"] * 62 + ["uchar"])
        refused("lacks the required properties \\['rot_3'\\]", names=names[:-1], rows=rows[:, :-1])
        refused("lacks the required properties \\['x', 'opacity'\\]", names=[n for n in names if n not in ("x", "opacity")],
                rows=rows[:, :60])
        refused("the first element is 'face 5', not 'vertex'", first="face")
        refused("the body holds 1240 bytes, the header says 3720", n=15)
        refused("f_rest_\\* must be", names=names[:20] + names[54:], rows=np.concatenate([rows[:, :20], rows[:, 54:]], 1))
        with open(path, "wb") as f:
            f.write(b"not a ply\n")
        with pytest.raises(ValueError, match="not a PLY file"):
            ply.read_ply(path)
        with open(path, "wb") as f:
            f.write(b"ply\nformat binary_little_endian 1.0\nelement vertex 1\nproperty float x\n")
        with pytest.raises(ValueError, match="no end_header"):
            ply.read_ply(path)
