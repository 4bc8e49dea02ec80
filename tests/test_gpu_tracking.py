"""Point tracking through the learned motion (rdg_track_attrs, rdg_track_project, engine.track, SplatTrainStep.track_maps /
track_points) and PCK-T (metrics.pck).

Yardsticks: the blended map S_m is bit-identical to engine.render_forward of the source view with colors_precomp = the
target-time centres rdg_track_attrs itself wrote (same records, same bins, same blend), and its alpha to render_views'; the
centres are held to a float64 restatement of the deformation, S_m to the oracle, the projection to a float64 restatement,
and the whole chain to a closed form (a scene that moves rigidly, seen by a camera that moves with it)."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from test_checkpoint import _cpu_step
from test_gpu_metrics import _same, _snapshot

# largest T whose table rows rdg_track_attrs stages in shared memory (RDG_TRACK_TABLE_MAX in track.cu)
TABLE_SMEM_MAX = 137
IMG_TOL = 1e-4


def _bits(t):
    """float32 tensor as int32 bits: NaN == NaN, for bit-identity checks of outputs that hold NaN"""
    return t.contiguous().view(torch.int32)


# ================================================================ CPU ==

def test_abi_refuses_bad_arguments_without_a_gpu():
    from rodygs_b200 import _lib
    lib = _lib.load()
    buf = (C.c_float * 64)()
    a = C.addressof(buf)
    scene, geom = _lib.RdgScene(), _lib.RdgGeom()
    scene.n_static = 4

    def attrs(sc=scene, gm=geom, bt=None):
        return lib.rdg_track_attrs(None if sc is None else C.byref(sc), bt, None if gm is None else C.byref(gm), None, None)

    assert attrs(sc=None) == -1 and b"null argument" in lib.rdg_last_error()
    assert attrs(gm=None) == -1 and b"null argument" in lib.rdg_last_error()
    scene.basis_t = a
    assert attrs() == -1 and b"basis_t must be NULL" in lib.rdg_last_error()
    scene.basis_t = None
    scene.n_static = -1
    assert attrs() == -1 and b"negative count" in lib.rdg_last_error()
    scene.n_static = 4
    assert attrs() == -1 and b"null geometry buffer" in lib.rdg_last_error()
    geom.radii = geom.p1 = a
    assert attrs() == -1 and b"null geometry buffer" in lib.rdg_last_error()      # p2 missing
    geom.p2 = a
    assert attrs() == -1 and b"null static parameter" in lib.rdg_last_error()
    scene.n_static, scene.n_dynamic, scene.raw, scene.use_deform, scene.num_basis, scene.num_times = 0, 4, 1, 1, 16, 5
    scene.dy.xyz = scene.motion_coeff = scene.time_ind = scene.table = a
    assert attrs() == -1 and b"null deformation input" in lib.rdg_last_error()    # basis_t_target missing
    scene.num_basis = 17
    assert attrs(bt=a) == -1 and b"num_basis" in lib.rdg_last_error()
    scene.n_dynamic = 0
    assert attrs() == 0                                                            # nothing to do: no launch

    def project(S=a, A=a, M=2, H=8, W=8, vm=a, pm=a, pts=None, P=0, xy=a, d=a):
        return lib.rdg_track_project(S, A, M, H, W, vm, pm, pts, P, xy, d, None, None)

    for kw in ({"S": None}, {"A": None}, {"vm": None}, {"pm": None}, {"xy": None}, {"d": None}):
        assert project(**kw) == -1 and b"null argument" in lib.rdg_last_error(), kw
    for kw in ({"H": 0}, {"W": 0}, {"H": -3}, {"W": -1}):
        assert project(**kw) == -1 and b"empty image" in lib.rdg_last_error(), kw
    for M in (0, -1, 65536):
        assert project(M=M) == -1 and b"M must be" in lib.rdg_last_error(), M
    for pts in (None, a):
        assert project(pts=pts, P=-1) == -1 and b"negative point count" in lib.rdg_last_error()
    assert project(pts=a, P=0) == 0                                                # no query point: no launch


def test_track_checks_its_arguments_on_the_host():
    step = _cpu_step(n=50)
    M = 3
    vm, pm, bt = torch.eye(4), torch.eye(4), torch.zeros(16, 7)
    vms, pms, bts = torch.eye(4).repeat(M, 1, 1), torch.eye(4).repeat(M, 1, 1), torch.zeros(M, 16, 7)
    pts = torch.zeros(5, 2)
    for fn, extra in ((step.track_maps, ()), (step.track_points, (pts,))):
        name = fn.__name__
        with pytest.raises(ValueError, match=f"{name}: target_viewmats must be a \\[M, 4, 4\\] tensor with M >= 1"):
            fn(vm, pm, 0.5, 0.5, bt, torch.zeros(0, 4, 4), pms, bts, *extra)
        with pytest.raises(ValueError, match="M >= 1"):
            fn(vm, pm, 0.5, 0.5, bt, None, pms, bts, *extra)
        with pytest.raises(ValueError, match="M >= 1"):
            fn(vm, pm, 0.5, 0.5, bt, torch.eye(4), pms, bts, *extra)
        with pytest.raises(ValueError, match="viewmat must be a contiguous float32 tensor of shape \\(4, 4\\)"):
            fn(vm.double(), pm, 0.5, 0.5, bt, vms, pms, bts, *extra)
        with pytest.raises(ValueError, match="viewmat must be"):
            fn(vm.t(), pm, 0.5, 0.5, bt, vms, pms, bts, *extra)                   # not contiguous
        with pytest.raises(ValueError, match="projmat must be"):
            fn(vm, pm[:3], 0.5, 0.5, bt, vms, pms, bts, *extra)
        with pytest.raises(ValueError, match="target_projmats must be"):
            fn(vm, pm, 0.5, 0.5, bt, vms, pms[:2], bts, *extra)
        with pytest.raises(ValueError, match="target_viewmats must be"):
            fn(vm, pm, 0.5, 0.5, bt, vms.double(), pms, bts, *extra)
        with pytest.raises(ValueError, match="basis_t must be"):
            fn(vm, pm, 0.5, 0.5, None, vms, pms, bts, *extra)
        with pytest.raises(ValueError, match="basis_t must be"):
            fn(vm, pm, 0.5, 0.5, bt[:8], vms, pms, bts, *extra)
        with pytest.raises(ValueError, match="target_basis_ts must be"):
            fn(vm, pm, 0.5, 0.5, bt, vms, pms, bts[:2], *extra)
        with pytest.raises(ValueError, match="target_basis_ts must be"):
            fn(vm, pm, 0.5, 0.5, bt, vms, pms, None, *extra)
        if torch.cuda.is_available():
            with pytest.raises(ValueError, match="viewmat must be .* on cpu, got .* cuda"):
                fn(vm.cuda(), pm, 0.5, 0.5, bt, vms, pms, bts, *extra)
    for bad in (None, torch.zeros(5, 3), torch.zeros(10), torch.zeros(5, 2, dtype=torch.float64), torch.zeros(2, 5).t()):
        with pytest.raises(ValueError, match="points must be"):
            step.track_points(vm, pm, 0.5, 0.5, bt, vms, pms, bts, bad)


def test_track_kernels_do_not_spill():
    """`-Xptxas -v` of track.cu (its own -fmad=false flags): no spills and no stack frame in any of its kernels."""
    from rodygs_b200 import build
    with tempfile.TemporaryDirectory() as tmp:
        r = subprocess.run([build._nvcc(), *build.ARCH, *build.COMMON, *build.SOURCES["track.cu"], "-Xptxas", "-v", "-c",
                            os.path.join(build.CSRC, "track.cu"), "-o", os.path.join(tmp, "track.o")],
                           capture_output=True, text=True, check=True)
    assert build.SOURCES["track.cu"] == ["-fmad=false"]
    info, name = {}, None
    for line in r.stderr.splitlines():
        hit = re.search(r"Compiling entry function '(\w+)'", line)
        if hit:
            name = hit.group(1)
        elif name and "spill" in line:
            info[name] = line.strip()
    assert len(info) == 3 and sum("track_attrs_kernel" in n for n in info) == 1, sorted(info)
    for n, line in info.items():
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in line, (n, line)


def _pck_numpy(pred, gt, vis, H, W, ratio=0.05):
    out = []
    for b in range(pred.shape[0]):
        n = hits = 0
        for p in range(pred.shape[1]):
            if not vis[b, p]:
                continue
            n += 1
            d = np.sqrt(np.sum((pred[b, p].astype(np.float64) - gt[b, p].astype(np.float64)) ** 2))
            hits += bool(d < ratio * max(H, W))
        out.append(hits / n if n else np.nan)
    return np.array(out)


def test_pck_against_numpy_and_closed_forms():
    from rodygs_b200.metrics import pck
    g = torch.Generator().manual_seed(0)
    H, W = 480, 640
    gt = torch.rand(6, 40, 2, generator=g) * torch.tensor([W, H])
    pred = gt + 40.0 * torch.randn(6, 40, 2, generator=g)
    pred[1, 3] = float("nan")
    vis = torch.rand(6, 40, generator=g) < 0.7
    vis[4] = False
    got = pck(pred, gt, vis, H, W)
    ref = _pck_numpy(pred.numpy(), gt.numpy(), vis.numpy(), H, W)
    assert got.dtype == torch.float64 and got.shape == (6,)
    assert np.allclose(got.numpy(), ref, equal_nan=True, rtol=0, atol=1e-15)
    assert torch.equal(pck(pred, gt, vis.float(), H, W).nan_to_num(-1), got.nan_to_num(-1))   # numeric visibility
    assert 0 < got[0] < 1 and torch.isnan(got[4]) and not torch.isnan(got[1])
    one = torch.ones(1, 40, dtype=torch.bool)
    assert pck(gt[:1], gt[:1], one, H, W).item() == 1.0                                 # exact
    direction = torch.nn.functional.normalize(torch.randn(1, 40, 2, generator=g, dtype=torch.float64), dim=-1)
    for frac, want in ((0.049, 1.0), (0.051, 0.0)):
        shifted = gt[:1].double() + frac * max(H, W) * direction
        assert pck(shifted, gt[:1], one, H, W).item() == want, frac
        assert pck(shifted, gt[:1], one, W, H).item() == want, frac                    # the longer side, either way round
    assert pck(gt[:1], gt[:1], one, H, W, ratio=1e-9).item() == 1.0                     # strictly within: 0 < thr
    nan_pred = gt[:1].clone()
    nan_pred[0, :10] = float("nan")
    assert pck(nan_pred, gt[:1], one, H, W).item() == 0.75                              # NaN counts as wrong
    part = one.clone()
    part[0, :10] = False
    assert pck(nan_pred, gt[:1], part, H, W).item() == 1.0                              # invisible points excluded
    assert torch.isnan(pck(gt[:1], gt[:1], torch.zeros(1, 40, dtype=torch.bool), H, W)).all()
    with pytest.raises(ValueError, match="pck: pred and gt must be"):
        pck(pred, gt[:, :5], vis, H, W)
    with pytest.raises(ValueError, match="pck: pred and gt must be"):
        pck(pred, gt, vis[:, :5], H, W)
    with pytest.raises(ValueError, match="positive"):
        pck(pred, gt, vis, 0, W)


# ================================================================ GPU ==

def _make_step(N, H, W, T=6, sh_degree=3, dynamic_fraction=0.5, seed=3):
    from rodygs_b200 import synthetic
    from rodygs_b200.trainer import SplatTrainStep
    scene = synthetic.to_device(synthetic.make_scene(N, H, W, T, seed=seed, dynamic_fraction=dynamic_fraction), "cuda")
    return SplatTrainStep(scene, H, W, sh_degree=sh_degree, w_pearson=0.0)


def _cams(step, V, seed=0):
    """V cameras around the scene and their B(t) = a table row plus noise (a time between the frames)."""
    from rodygs_b200 import synthetic
    cams = [synthetic.make_camera(v, max(V, 2), step.H, step.W, step.T) for v in range(V)]
    vms = torch.stack([c.world_view_transform.t().contiguous() for c in cams]).cuda()
    pms = torch.stack([c.projection_matrix.t().contiguous() for c in cams]).cuda()
    g = torch.Generator(device="cuda").manual_seed(seed)
    bts = torch.stack([step.p("table")[c.time_index] for c in cams])
    bts = (bts + 0.01 * torch.randn(bts.shape, device="cuda", generator=g)).contiguous()
    return vms, pms, cams[0].tanfovx, cams[0].tanfovy, bts


def _track(step, vms, pms, fx, fy, bts, src=0, points=None, keep_maps=True):
    """engine.track of source view `src` into every view, as SplatTrainStep._track calls it"""
    from rodygs_b200 import engine
    scene, view = step._scene_view(vms[src], pms[src], fx, fy, None)
    dyn = step.nd > 0
    return engine.track(scene, view, bts[src] if dyn else None, vms, pms, bts if dyn else None, points, keep_maps=keep_maps)


def _positions64(step, bt):
    """float64 restatement of mu_k(t_m) for B(t_m) = bt, and the size of its terms (for the error bound)"""
    xyz = torch.cat([step.p("static.xyz"), step.p("dynamic.xyz")]).double()
    scale = torch.zeros_like(xyz).copy_(xyz.abs())
    if step.nd > 0:
        c = step.p("motion_coeff").view(step.nd, step.num_basis).double()
        diff = bt.double()[None] - step.p("table").double()[step.time_ind.long()]         # [nd, K, 7]
        terms = c[:, :, None] * diff[:, :, 0:3]
        xyz[step.ns:] += step.spatial_lr_scale * terms.sum(1)
        scale[step.ns:] += step.spatial_lr_scale * terms.abs().sum(1)
    return xyz, scale


def _assert_identical(step, M, seed=0):
    """S_m == render_forward(colors_precomp = positions_out of target m, bg 0) colour, alpha == render_views' alpha,
    positions_out against float64, and track_maps == engine.track."""
    from rodygs_b200 import engine
    vms, pms, fx, fy, bts = _cams(step, M, seed)
    xy, depth, alpha, S, pos = _track(step, vms, pms, fx, fy, bts)
    assert xy.shape == (M, 2, step.H, step.W) and depth.shape == (M, 1, step.H, step.W) and alpha.shape == (1, step.H, step.W)
    ref_alpha = step.render_views(vms[:1], pms[:1], fx, fy, bts[:1] if step.nd > 0 else None)[2][0]
    assert torch.equal(alpha, ref_alpha) and (alpha > 0).any()
    zero = torch.zeros(3, device="cuda")
    for m in range(M):
        scene, view = step._scene_view(vms[0], pms[0], fx, fy, bts[0] if step.nd > 0 else None)
        scene.colors_precomp, view.bg = pos[m], zero
        color, _, a, radii, _ = engine.render_forward(scene, view, keep_for_backward=False)
        assert torch.equal(S[m], color), (m, (S[m] != color).sum().item())
        assert torch.equal(a, alpha)
        ref, scale = _positions64(step, bts[m])
        err = (pos[m].double() - ref).abs()
        assert (err <= 1e-6 * scale).all(), (m, (err / scale).max().item())
    assert (radii > 0).any() and (radii == 0).any()                  # something visible, something culled
    got = step.track_maps(vms[0], pms[0], fx, fy, bts[0] if step.nd > 0 else None, vms, pms, bts if step.nd > 0 else None)
    for a, b in zip(got, (xy, depth, alpha)):
        assert torch.equal(_bits(a), _bits(b))
    hit = alpha[0] > 0
    assert torch.isnan(xy[:, :, ~hit]).all() and torch.isnan(depth[:, :, ~hit]).all()
    assert not torch.isnan(xy[:, :, hit]).any() and not torch.isnan(depth[:, :, hit]).any()
    # target 0 is the source camera at the source time: a pixel's track lands within a footprint of itself
    grid = torch.stack(torch.meshgrid(torch.arange(step.W, device="cuda"), torch.arange(step.H, device="cuda"), indexing="xy"))
    assert (xy[0, :, hit] - grid[:, hit]).abs().median() < 4.0


@pytest.mark.gpu
@pytest.mark.parametrize("dynamic_fraction,T,sh_degree,M", [
    (0.5, 6, 3, 8), (0.5, TABLE_SMEM_MAX, 0, 1), (0.5, TABLE_SMEM_MAX + 1, 3, 11), (0.0, 6, 3, 3), (1.0, 6, 0, 8),
    (1.0, TABLE_SMEM_MAX, 3, 3), (1.0, TABLE_SMEM_MAX + 1, 0, 3)])
def test_blended_map_is_the_render_of_the_target_time_centres(dynamic_fraction, T, sh_degree, M):
    """97x131 (neither side a multiple of the 16-pixel tile), 20 001 Gaussians (not a multiple of the 256-Gaussian chunk,
    1 % behind the near plane), both table paths, SH degrees 0 and 3, M = 1, 3, 8 and 11 (a pass of 8 and a pass of 3)."""
    _assert_identical(_make_step(20_001, 97, 131, T=T, sh_degree=sh_degree, dynamic_fraction=dynamic_fraction), M, seed=M)


@pytest.mark.gpu
def test_blended_map_against_the_oracle():
    """S_m against oracle.splat_oracle.rasterize on the activated values the source render used, with colors_precomp = the
    float64 target-time centres and a zero background: max-abs <= 1e-4 of the map's largest value.  Where float32 cannot
    resolve that (a weight at the 1/255 threshold), the float32 oracle's own distance to float64 is the yardstick."""
    import helpers
    from oracle import splat_oracle as so
    from rodygs_b200 import engine, synthetic
    step = _make_step(4_001, 97, 131, T=6)
    vms, pms, fx, fy, bts = _cams(step, 3, seed=1)
    _, _, _, S, pos = _track(step, vms, pms, fx, fy, bts)
    engine.config.debug_activated = True
    try:
        scene, view = step._scene_view(vms[0], pms[0], fx, fy, bts[0])
        state = engine.render_forward(scene, view)[4]
        act = state.geom["dbg_activated"].cpu()
    finally:
        engine.config.debug_activated = False
    cam = synthetic.make_camera(0, 3, step.H, step.W, step.T)
    st32 = helpers.oracle_settings(cam, torch.zeros(3), 0)
    st64 = so.Settings(step.H, step.W, fx, fy, torch.zeros(3, dtype=torch.float64), 1.0,
                       pms[0].cpu().double(), 0)
    vm = vms[0].cpu()
    for m in range(3):
        ref64 = _positions64(step, bts[m])[0].cpu()
        o32 = so.rasterize(act[:, 0:3].contiguous(), None, None, pos[m].cpu(), act[:, 10:11].contiguous(),
                           act[:, 3:6].contiguous(), act[:, 6:10].contiguous(), vm, st32)
        o64 = so.rasterize(act[:, 0:3].double(), None, None, ref64, act[:, 10:11].double(), act[:, 3:6].double(),
                           act[:, 6:10].double(), vm.double(), st64)
        tol = IMG_TOL * max(1.0, S[m].abs().max().item())
        err64 = (S[m].cpu().double() - o64.color).abs().max().item()
        noise = (o32.color.double() - o64.color).abs().max().item()
        assert err64 <= tol or err64 <= 1.5 * noise + tol, (m, err64, noise, tol)


def _project64(S, A, vms, pms, H, W):
    """float64 restatement of the normalisation and projection on maps S [M, 3, ...], A [...]"""
    X = S.double() / A.double()
    out_xy, out_d = [], []
    for m in range(S.shape[0]):
        V, P = vms[m].double().t(), pms[m].double().t()
        Xh = torch.cat([X[m].reshape(3, -1), torch.ones(1, X[m][0].numel(), dtype=torch.float64, device=X.device)])
        v = V @ Xh
        c = P @ v
        ndc = c[:2] / (c[3] + 1e-7)
        px, py = ((ndc[0] + 1) * W - 1) / 2, ((ndc[1] + 1) * H - 1) / 2
        out_xy.append(torch.stack([px, py]))
        out_d.append(v[2])
    return torch.stack(out_xy), torch.stack(out_d)


def _bilinear64(img, x, y):
    """img [C, H, W] sampled at (x, y) between pixel centres, clamped to the image, as a + f (b - a), in float64"""
    Cc, H, W = img.shape
    img = img.double()
    x, y = x.double().clamp(0, W - 1), y.double().clamp(0, H - 1)
    x0, y0 = x.floor().long(), y.floor().long()
    x1, y1 = (x0 + 1).clamp(max=W - 1), (y0 + 1).clamp(max=H - 1)
    fx, fy = x - x0, y - y0

    def lerp(a, b, f):
        return a + f * (b - a)

    top = lerp(img[:, y0, x0], img[:, y0, x1], fx)
    bot = lerp(img[:, y1, x0], img[:, y1, x1], fx)
    return lerp(top, bot, fy)


@pytest.mark.gpu
def test_projection_dense_and_sparse_against_float64():
    """rdg_track_project on random maps of points in front of the targets (A in [0.2, 1], 0 in a tenth of the pixels):
    dense and sparse (points across the image, on its edges and beyond them: clamped) within 1e-3 px and depth within 1e-5
    relative of a float64 restatement, NaN exactly where A == 0; sparse at integer points has the dense pixels' bits."""
    from rodygs_b200 import _lib, synthetic
    lib = _lib.load()
    H, W, M = 97, 131, 5
    g = torch.Generator(device="cuda").manual_seed(4)
    cams = [synthetic.make_camera(v, M, H, W, 6) for v in range(M)]
    vms = torch.stack([c.world_view_transform.t().contiguous() for c in cams]).cuda()
    pms = torch.stack([c.projection_matrix.t().contiguous() for c in cams]).cuda()
    A = 0.2 + 0.8 * torch.rand(H, W, device="cuda", generator=g)
    A[torch.rand(H, W, device="cuda", generator=g) < 0.1] = 0.0
    A[0, 0] = A[H - 1, W - 1] = 0.0
    X = torch.stack([3.0 * torch.rand(M, H, W, device="cuda", generator=g) - 1.5,
                     2.0 * torch.rand(M, H, W, device="cuda", generator=g) - 1.0,
                     2.5 + 4.0 * torch.rand(M, H, W, device="cuda", generator=g)], 1)
    S = (X * A).contiguous()
    stream = _lib.stream_ptr()
    xy, depth = torch.empty(M, 2, H, W, device="cuda"), torch.empty(M, 1, H, W, device="cuda")
    _lib.check(lib.rdg_track_project(S.data_ptr(), A.data_ptr(), M, H, W, vms.data_ptr(), pms.data_ptr(), None, 0,
                                     xy.data_ptr(), depth.data_ptr(), None, stream))
    ref_xy, ref_d = _project64(S, A, vms, pms, H, W)
    hole = (A == 0).reshape(-1)
    xy_f, d_f = xy.reshape(M, 2, -1), depth.reshape(M, -1)
    assert torch.isnan(xy_f[:, :, hole]).all() and torch.isnan(d_f[:, hole]).all()
    assert (xy_f[:, :, ~hole].double() - ref_xy[:, :, ~hole]).abs().max() <= 1e-3
    assert ((d_f[:, ~hole].double() - ref_d[:, ~hole]).abs() / ref_d[:, ~hole].abs()).max() <= 1e-5
    # sparse: random points over and beyond the image, the four corners and edge midpoints, one NaN point
    P = 600
    pts = torch.stack([torch.rand(P, device="cuda", generator=g) * (W + 6) - 3,
                       torch.rand(P, device="cuda", generator=g) * (H + 6) - 3], 1)
    edges = torch.tensor([[0, 0], [W - 1, 0], [0, H - 1], [W - 1, H - 1], [W - 1, 40.5], [70.25, H - 1], [-5, 30.5],
                          [W + 9, 20.75], [15.5, -2], [33.75, H + 4]], dtype=torch.float32, device="cuda")
    pts = torch.cat([pts, edges, torch.tensor([[float("nan"), 3.0]], device="cuda")]).contiguous()
    P = pts.shape[0]
    sxy, sd, sa = torch.empty(M, P, 2, device="cuda"), torch.empty(M, P, device="cuda"), torch.empty(P, device="cuda")
    _lib.check(lib.rdg_track_project(S.data_ptr(), A.data_ptr(), M, H, W, vms.data_ptr(), pms.data_ptr(), pts.data_ptr(), P,
                                     sxy.data_ptr(), sd.data_ptr(), sa.data_ptr(), stream))
    Ai = _bilinear64(A[None], pts[:-1, 0], pts[:-1, 1])[0]
    Si = torch.stack([_bilinear64(S[m], pts[:-1, 0], pts[:-1, 1]) for m in range(M)])
    rxy, rd = _project64(Si, Ai, vms, pms, H, W)
    ok = Ai > 0
    assert ok.sum() > P // 2 and (~ok).sum() >= 2
    assert (sa[:-1].double() - Ai).abs().max() <= 1e-6
    assert (sxy[:, :-1][:, ok].double() - rxy.transpose(1, 2)[:, ok]).abs().max() <= 1e-3
    assert ((sd[:, :-1][:, ok].double() - rd[:, ok]).abs() / rd[:, ok].abs()).max() <= 1e-5
    assert torch.isnan(sxy[:, :-1][:, ~ok]).all() and torch.isnan(sd[:, :-1][:, ~ok]).all()
    assert torch.isnan(sxy[:, -1]).all() and torch.isnan(sd[:, -1]).all() and torch.isnan(sa[-1])
    # integer points (every pixel of a few rows and columns, the corners included): the dense pixels' bits
    ys, xs = torch.meshgrid(torch.tensor([0, 1, 48, H - 1]), torch.arange(W), indexing="ij")
    ys2, xs2 = torch.meshgrid(torch.arange(H), torch.tensor([0, 77, W - 1]), indexing="ij")
    ix = torch.cat([xs.reshape(-1), xs2.reshape(-1)]).cuda()
    iy = torch.cat([ys.reshape(-1), ys2.reshape(-1)]).cuda()
    ipts = torch.stack([ix, iy], 1).float().contiguous()
    Q = ipts.shape[0]
    qxy, qd, qa = torch.empty(M, Q, 2, device="cuda"), torch.empty(M, Q, device="cuda"), torch.empty(Q, device="cuda")
    _lib.check(lib.rdg_track_project(S.data_ptr(), A.data_ptr(), M, H, W, vms.data_ptr(), pms.data_ptr(), ipts.data_ptr(), Q,
                                     qxy.data_ptr(), qd.data_ptr(), qa.data_ptr(), stream))
    assert torch.equal(_bits(qxy), _bits(xy[:, :, iy, ix].transpose(1, 2)))
    assert torch.equal(_bits(qd), _bits(depth[:, 0, iy, ix]))
    assert torch.equal(qa, A[iy, ix])


@pytest.mark.gpu
def test_track_points_at_integer_points_is_track_maps():
    """Through SplatTrainStep: track_points at integer pixels returns track_maps' bits there (alpha included)."""
    step = _make_step(20_001, 97, 131, T=12)
    vms, pms, fx, fy, bts = _cams(step, 4, seed=2)
    xy, depth, alpha = step.track_maps(vms[0], pms[0], fx, fy, bts[0], vms, pms, bts)
    g = torch.Generator(device="cuda").manual_seed(3)
    ix = torch.randint(0, step.W, (500,), device="cuda", generator=g)
    iy = torch.randint(0, step.H, (500,), device="cuda", generator=g)
    pts = torch.stack([ix, iy], 1).float().contiguous()
    pxy, pd, pa = step.track_points(vms[0], pms[0], fx, fy, bts[0], vms, pms, bts, pts)
    assert pxy.shape == (4, 500, 2) and pd.shape == (4, 500) and pa.shape == (500,)
    assert torch.equal(_bits(pxy), _bits(xy[:, :, iy, ix].transpose(1, 2)))
    assert torch.equal(_bits(pd), _bits(depth[:, 0, iy, ix]))
    assert torch.equal(pa, alpha[0, iy, ix])
    empty = step.track_points(vms[0], pms[0], fx, fy, bts[0], vms, pms, bts, torch.zeros(0, 2, device="cuda"))
    assert empty[0].shape == (4, 0, 2) and empty[1].shape == (4, 0) and empty[2].shape == (0,)


def _translated(vm_glm, delta):
    """glm-storage view matrix of the camera moved by delta along with the scene: V' X = V (X - delta)"""
    V = vm_glm.double().t()
    Tm = torch.eye(4, dtype=torch.float64, device=V.device)
    Tm[:3, 3] = -delta
    return (V @ Tm).t().contiguous().float()


@pytest.mark.gpu
def test_rigid_motion_known_answer_and_pck():
    """Every dynamic Gaussian with the same coefficient row moves by the same delta = s sum_b c_b (B(t_m) - B(t_s))[0:3].
    A target camera moved by delta at t_m then sees what the source camera sees at t_s: the tracks equal the same-time
    tracks within 1e-3 px.  PCK-T of keypoints taken from those tracks is 1; shifted past the threshold it is 0."""
    from rodygs_b200.metrics import pck
    step = _make_step(20_000, 97, 131, T=6, dynamic_fraction=1.0)
    g = torch.Generator(device="cuda").manual_seed(8)
    row = 0.5 * torch.randn(step.num_basis, device="cuda", generator=g)
    step.p("motion_coeff").view(step.nd, step.num_basis).copy_(row.expand(step.nd, -1))
    vms, pms, fx, fy, bts = _cams(step, 3, seed=5)
    delta = [step.spatial_lr_scale * (row.double()[:, None] * (bts[m].double() - bts[0].double())[:, 0:3]).sum(0)
             for m in range(3)]
    assert min(d.norm().item() for d in delta[1:]) > 0.02                       # a real motion
    moved = torch.stack([_translated(vms[0], delta[m]) for m in range(3)])
    same = step.track_maps(vms[0], pms[0], fx, fy, bts[0], vms[:1].expand(3, 4, 4).contiguous(), pms[:1].expand(3, 4, 4).contiguous(),
                           bts[:1].expand(3, -1, -1).contiguous())
    got = step.track_maps(vms[0], pms[0], fx, fy, bts[0], moved, pms[:1].expand(3, 4, 4).contiguous(), bts)
    hit = got[2][0] > 0
    assert hit.sum() > 1000
    assert torch.equal(got[2], same[2])
    assert (got[0][:, :, hit] - same[0][:, :, hit]).abs().max() <= 1e-3
    assert ((got[1][:, :, hit] - same[1][:, :, hit]).abs() / same[1][:, :, hit].abs()).max() <= 1e-5
    # keypoints: integer pixels with alpha > 0.5, ground truth = the same-time tracks there
    iy, ix = torch.nonzero(got[2][0] > 0.5, as_tuple=True)
    sel = torch.randperm(iy.numel(), device="cuda", generator=g)[:300]
    iy, ix = iy[sel], ix[sel]
    pts = torch.stack([ix, iy], 1).float().contiguous()
    pred = step.track_points(vms[0], pms[0], fx, fy, bts[0], moved, pms[:1].expand(3, 4, 4).contiguous(), bts, pts)[0]
    gt = same[0][:, :, iy, ix].transpose(1, 2)
    vis = torch.ones(3, pts.shape[0], dtype=torch.bool, device="cuda")
    assert torch.equal(pck(pred, gt, vis, step.H, step.W), torch.ones(3, dtype=torch.float64, device="cuda"))
    shift = torch.tensor([0.06 * max(step.H, step.W), 0.0], device="cuda")
    assert torch.equal(pck(pred + shift, gt, vis, step.H, step.W), torch.zeros(3, dtype=torch.float64, device="cuda"))


def _camera_snapshot(step):
    return {k: (v.clone() if torch.is_tensor(v) else v) for k, v in step.cameras.items()}


@pytest.mark.gpu
def test_tracking_leaves_the_training_state_alone():
    """After forward_backward (+ exchange_grads(defer_sh=True)), densification statistics, both optimisers and a camera table:
    every piece of training state is bit-identical after track_maps and track_points (the source camera a learned one,
    through camera_viewmatrix), the duplicate capacity is untouched, and two calls return the same bits."""
    from rodygs_b200 import engine
    from rodygs_b200.optim import CameraLRs, GaussianLRs
    step = _make_step(20_000, 176, 208)
    step.attach_optimizer("static", GaussianLRs())
    step.attach_optimizer("dynamic", GaussianLRs(scaling_lr=0.001, motion_coeff_lr=1.6e-4))
    step.enable_densification("static")
    step.enable_densification("dynamic")
    step.enable_factored_exchange(views_per_rank=1, world_size=1)
    vms, pms, fx, fy, bts = _cams(step, 9)
    step.enable_camera_learning(vms[:2].contiguous(), CameraLRs(1e-4, 1e-4))
    gt = torch.rand(3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    for it in (1, 2):
        step.forward_backward(vms[0], pms[0], fx, fy, bts[0], gt, None, dcolor_slot=0)
        step.exchange_grads(vms[:1].contiguous(), bts[:1].contiguous(), defer_sh=True)
        if it == 1:
            for tag in ("static", "dynamic"):
                step.add_densification_stats(tag)
                step.optimizer_step(tag, it)
    torch.cuda.synchronize()
    before, cams = _snapshot(step), _camera_snapshot(step)
    cap = {k: dict(v) for k, v in engine._capacity.items()}
    gen = torch.Generator(device="cuda").manual_seed(7)           # not the global generator: it is training state
    pts = (torch.rand(50, 2, device="cuda", generator=gen) * torch.tensor([207.0, 175.0], device="cuda")).contiguous()
    args = (step.camera_viewmatrix(1), pms[1], fx, fy, bts[1], vms, pms, bts)
    first = step.track_maps(*args) + step.track_points(*args, pts)
    second = step.track_maps(*args) + step.track_points(*args, pts)
    torch.cuda.synchronize()
    after = _snapshot(step)
    assert all(torch.equal(_bits(a), _bits(b)) for a, b in zip(first, second))
    assert after["last_state"] is before["last_state"] and after["deferred"] is before["deferred"]
    assert all(x is y for x, y in zip(after["last_outputs"], before["last_outputs"]))
    for key in before:
        assert _same(before[key], after[key]), key
    assert _same(cams, _camera_snapshot(step))
    assert engine._capacity.keys() == cap.keys()
    for k, st in engine._capacity.items():
        assert st["cap"] == cap[k]["cap"] and st["pending"] is cap[k]["pending"]
    for tag in ("static", "dynamic"):
        step.add_densification_stats(tag)
        step.optimizer_step(tag, 2)
    assert not step._deferred["pending"]


@pytest.mark.gpu
def test_a_pending_sync_free_count_stays_for_the_training_step():
    """Under config.sync_free the training step leaves its duplicate count unread.  Tracking neither reads nor clears it:
    here the pending record claims buffers far smaller than the frame needed, track_maps still returns the same bits as
    without a pending count, and the next forward_backward raises the overflow that belongs to it."""
    from rodygs_b200 import engine
    step = _make_step(20_000, 176, 208)
    vms, pms, fx, fy, bts = _cams(step, 3)
    ref = step.track_maps(vms[0], pms[0], fx, fy, bts[0], vms, pms, bts)
    gt = torch.rand(3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(6))
    saved = engine.config.sync_free
    engine.config.sync_free = True
    try:
        step.forward_backward(vms[0], pms[0], fx, fy, bts[0], gt, None)
        st = engine._cap_state(step.params.device, step.ns + step.nd)
        host, ev, _ = st["pending"]
        st["pending"] = pending = (host, ev, 1)          # as if that frame had been truncated
        cap = st["cap"]
        got = step.track_maps(vms[0], pms[0], fx, fy, bts[0], vms, pms, bts)
        assert st["pending"] is pending and st["cap"] == cap
        assert all(torch.equal(_bits(a), _bits(b)) for a, b in zip(got, ref))
        with pytest.raises(RuntimeError, match="truncated"):
            step.forward_backward(vms[0], pms[0], fx, fy, bts[0], gt, None)
    finally:
        engine.config.sync_free = saved
        engine._cap_state(step.params.device, step.ns + step.nd)["pending"] = None
