"""CUDA path against frozen / full-density / adversarial cases (VERDICT r01 "harden rasterizer parity"):
  * tests/golden/raster_small.npz - the oracle's outputs frozen on disk (no oracle call at all);
  * BASELINE.json config 1 exactly (10K Gaussians, 50 % dynamic, 256x256, 8 frames) through the fused path;
  * the density-matched window of the bench workload that bench.py's CPU arm times (62 745 Gaussians, 256x256, T = 100,
    736 list entries per tile against 723 at config 4);
  * an adversarial sweep for the sub-tile masks of the blend kernels (rdg_sub_mask decides which pixels are ever visited):
    radius 0.5 / 40 / 200 px, 100:1 anisotropy at random angles, opacity logits -5.5 / +6, centres up to two radii outside
    the image, scale_modifier 0.3 / 3.
Bars: integer outputs bit-exact, images 1e-4 max-abs, gradients 1e-3 (norm-wise for the large per-Gaussian tensors and
ELEMENT-wise, |a - b| <= 1e-3 |b| + 1e-5 max|b|, for dL/dV, dL/dtable, dL/dB(t), dL/dcoeff)."""
import math
import os

import numpy as np
import pytest
import torch

import helpers
from conftest import GOLDEN
from oracle import deform_oracle as do
from oracle import splat_oracle as so
from rodygs_b200 import engine, synthetic
from rodygs_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer

pytestmark = pytest.mark.gpu

IMG_TOL, GRAD_TOL = 1e-4, 1e-3


elementwise_ok = helpers.elementwise_ok
elementwise_vs_truth = helpers.elementwise_vs_truth


def normwise_vs_truth(got, ref32, ref64, tol=GRAD_TOL):
    """max|a - b| / max|b| <= tol against the float32 oracle, or as close to the float64 oracle as 1.5 x the float32 one."""
    e32 = helpers.rel_err(got.cpu(), ref32)
    if e32 <= tol:
        return True, e32, 0.0
    e64 = helpers.rel_err(got.double().cpu(), ref64)
    n64 = helpers.rel_err(ref32.double(), ref64)
    return e64 <= 1.5 * n64 + tol, e64, n64


@pytest.fixture(autouse=True)
def _reset():
    yield
    engine.config.sync_free = False
    engine.config.binning = "tiles"
    engine.config.debug_keep_unsorted = False
    engine.config.deterministic = False


def _boundary(acts, cam_vm, proj, tanfov, H, W, bg, deg, grads, mod=1.0):
    xyz, op, scl, rot, feat = [t.detach().clone().cuda().requires_grad_(True) for t in acts]
    vm = cam_vm.detach().clone().cuda().requires_grad_(True)
    m2 = torch.zeros(xyz.shape[0], 3, device="cuda", requires_grad=True)
    st = GaussianRasterizationSettings(H, W, tanfov[0], tanfov[1], bg.cuda(), mod, proj.cuda(), deg, False, False, True, True)
    out = GaussianRasterizer(st)(means3D=xyz, means2D=m2, shs=feat, colors_precomp=None, opacities=op, scales=scl,
                                 rotations=rot, cov3Ds_precomp=None, viewmatrix=vm)
    gc, gd, ga = [g.cuda() for g in grads]
    ((out[0] * gc).sum() + (out[1] * gd).sum() + (out[3] * ga).sum()).backward()
    g = {"means3D": xyz.grad, "means2D": m2.grad, "shs": feat.grad, "opacities": op.grad, "scales": scl.grad,
         "rotations": rot.grad, "viewmatrix": vm.grad}
    return out, g


def test_cuda_path_against_the_frozen_fixture():
    f = {k: torch.from_numpy(np.asarray(v)) for k, v in np.load(os.path.join(GOLDEN, "raster_small.npz")).items()}
    n, H, W, deg = [int(v) for v in f["meta"]]
    acts = (f["means3D"], f["opacities"], f["scales"], f["rotations"], f["shs"])
    tanfov = (float(f["tanfov"][0]), float(f["tanfov"][1]))
    for binning in ("tiles", "lsd"):
        engine.config.binning = binning
        out, g = _boundary(acts, f["viewmatrix"], f["projmatrix"], tanfov, H, W, f["bg"], deg,
                           (f["dL_dcolor"], f["dL_ddepth"], f["dL_dalpha"]))
        assert torch.equal(out[4].cpu(), f["radii"])
        assert (out[0].cpu() - f["color"]).abs().max() <= IMG_TOL
        assert (out[1].cpu() - f["depth"]).abs().max() <= IMG_TOL
        assert (out[3].cpu() - f["alpha"]).abs().max() <= IMG_TOL
        for k in ("means3D", "means2D", "shs", "opacities", "scales", "rotations"):
            err = helpers.rel_err(g[k].cpu(), f["g_" + k])
            assert err <= GRAD_TOL, f"{binning} grad {k}: {err:.3e}"
        ok, ratio = elementwise_ok(g["viewmatrix"], f["g_viewmatrix"])
        assert ok, f"{binning} dL/dV element-wise: {ratio:.2f} x the bound"
    # sorted keys / order / ranges of the frozen scene (engine level, both binning paths)
    xyz, op, scl, rot, feat = [t.cuda() for t in acts]
    scene = engine.SceneArgs(st=engine.SetArgs(xyz=xyz, scaling=scl, rotation=rot, opacity=op, sh_dc=feat, sh_rest=feat,
                                               sh_dc_stride=48, sh_rest_stride=48, sh_rest_offset=3), raw=False)
    view = engine.ViewArgs(H, W, tanfov[0], tanfov[1], 1.0, deg, f["viewmatrix"].cuda(), f["projmatrix"].cuda(), f["bg"].cuda())
    for binning in ("tiles", "lsd"):
        engine.config.binning = binning
        _, _, _, _, state = engine.render_forward(scene, view)
        D = int(state.num_rendered[0])
        assert D == f["keys"].numel()
        assert torch.equal(state.extras["keys_sorted"][:D].cpu(), f["keys"])
        assert torch.equal(state.vals_sorted[:D].cpu(), f["vals"])
        assert torch.equal(state.ranges.cpu(), f["ranges"])
        assert torch.equal(state.geom["tiles_touched"].cpu(), f["tiles_touched"])
        assert (state.final_T.cpu() - f["final_T"]).abs().max() <= IMG_TOL


def _chain(sc, cam, H, W, deg, up, bg, dt):
    """Reference chain on the CPU in dtype dt: activations -> deformation -> concat -> rasterize -> backward."""
    def leaf(t):
        return t.detach().clone().to(dt).requires_grad_(True)
    n = sc["static"]["xyz"].shape[0] + sc["dynamic"]["xyz"].shape[0]
    st = do.RawGaussians(**{k: leaf(v) for k, v in sc["static"].items()})
    dy = do.RawGaussians(**{k: leaf(v) for k, v in sc["dynamic"].items()})
    coeff, table = leaf(sc["motion_coeff"]), leaf(sc["table"])
    basis_t = leaf(sc["table"][cam.time_index])
    acts = do.assemble(st, dy, coeff.squeeze(1), basis_t, table, sc["time_ind"].long(), sc["spatial_lr_scale"], True)
    vm = leaf(cam.world_view_transform.t().contiguous())
    m2 = torch.zeros(n, 3, dtype=dt, requires_grad=True)
    xyz, op, scl, rot, feat = acts
    settings = so.Settings(H, W, cam.tanfovx, cam.tanfovy, bg.to(dt), 1.0, cam.projection_matrix.t().contiguous().to(dt), deg)
    orc = so.rasterize(xyz, m2, feat, None, op, scl, rot, vm, settings)
    ((orc.color * up[0].to(dt)).sum() + (orc.depth * up[1].to(dt)).sum() + (orc.alpha * up[2].to(dt)).sum()).backward()
    grads = {f"{tag}.{k}": getattr(obj, k).grad for tag, obj in (("static", st), ("dynamic", dy))
             for k in ("xyz", "scaling", "rotation", "opacity", "features_dc", "features_rest")}
    grads.update(means2D=m2.grad, viewmatrix=vm.grad, table=table.grad, basis_t=basis_t.grad, motion_coeff=coeff.grad)
    return orc, grads


ELEMENTWISE = ("viewmatrix", "table", "basis_t", "motion_coeff")


def _fused_vs_chain(sc, cam, H, W, deg=3, w_img=(1.0, 0.3, 0.2), seed=5, bg=None, truth64=False):
    """Fused path on raw parameters vs the reference chain on the CPU.  Returns (image error, radii mismatch fraction,
    {name: norm-wise error}, {name: (ok, ratio[, float32 oracle's ratio])} for the element-wise group, duplicates)."""
    from rodygs_b200.dynamic import GaussianParams, render_dynamic
    bg = torch.zeros(3) if bg is None else bg
    g = torch.Generator().manual_seed(seed)
    up = (w_img[0] * torch.randn(3, H, W, generator=g), w_img[1] * torch.randn(1, H, W, generator=g), w_img[2] * torch.randn(1, H, W, generator=g))
    orc, ref = _chain(sc, cam, H, W, deg, up, bg, torch.float32)
    ref64 = _chain(sc, cam, H, W, deg, up, bg, torch.float64)[1] if truth64 else None

    cst = GaussianParams(**{k: v.cuda().requires_grad_(True) for k, v in sc["static"].items()})
    cdy = GaussianParams(**{k: v.cuda().requires_grad_(True) for k, v in sc["dynamic"].items()})
    ccoeff = sc["motion_coeff"].cuda().requires_grad_(True)
    ctable = sc["table"].cuda().requires_grad_(True)
    cbasis = sc["table"][cam.time_index].cuda().requires_grad_(True)
    cvm = cam.world_view_transform.t().contiguous().cuda().requires_grad_(True)
    settings = GaussianRasterizationSettings(H, W, cam.tanfovx, cam.tanfovy, bg.cuda(), 1.0,
                                             cam.projection_matrix.t().contiguous().cuda(), deg, False, False, True, True)
    pkg = render_dynamic(cst, cdy, settings, cvm, ccoeff, cbasis, ctable, sc["time_ind"].cuda(), sc["spatial_lr_scale"], True)
    ((pkg["rendered_image"] * up[0].cuda()).sum() + (pkg["rendered_depth"] * up[1].cuda()).sum()
     + (pkg["rendered_alpha"] * up[2].cuda()).sum()).backward()
    img_err = max((pkg["rendered_image"].cpu() - orc.color).abs().max().item(),
                  (pkg["rendered_depth"].cpu() - orc.depth).abs().max().item(),
                  (pkg["rendered_alpha"].cpu() - orc.alpha).abs().max().item())
    radii_mismatch = (pkg["radii"].cpu() != orc.radii).float().mean().item()
    got = {f"{tag}.{k}": getattr(obj, k).grad for tag, obj in (("static", cst), ("dynamic", cdy))
           for k in ("xyz", "scaling", "rotation", "opacity", "features_dc", "features_rest")}
    got.update(means2D=pkg["viewspace_points"].grad, viewmatrix=cvm.grad, table=ctable.grad, basis_t=cbasis.grad, motion_coeff=ccoeff.grad)
    errs = {k: helpers.rel_err(got[k].cpu(), ref[k]) for k in got if k not in ELEMENTWISE}
    if truth64:
        elem = {k: elementwise_vs_truth(got[k], ref[k], ref64[k]) for k in ELEMENTWISE}
    else:
        elem = {k: elementwise_ok(got[k], ref[k]) for k in ELEMENTWISE}
    return img_err, radii_mismatch, errs, elem, int(orc.bn.keys.numel())


def _fused_forward_on_own_activations(sc, cam, H, W, deg=3):
    """Integer outputs bit-exact and images <= 1e-4 against the oracle evaluated on the activated values the fused kernel
    itself used (exp / sigmoid differ from the CPU's by ulps, which can flip a ceil() or a 1/255 threshold)."""
    dev = "cuda"
    engine.config.debug_activated = True
    try:
        def mk(d):
            return engine.SetArgs(xyz=d["xyz"].to(dev), scaling=d["scaling"].to(dev), rotation=d["rotation"].to(dev),
                                  opacity=d["opacity"].to(dev), sh_dc=d["features_dc"].to(dev), sh_rest=d["features_rest"].to(dev))
        scene = engine.SceneArgs(st=mk(sc["static"]), dy=mk(sc["dynamic"]), raw=True, use_deform=True,
                                 motion_coeff=sc["motion_coeff"].squeeze(1).contiguous().to(dev), time_ind=sc["time_ind"].to(dev),
                                 basis_t=sc["table"][cam.time_index].contiguous().to(dev), table=sc["table"].to(dev),
                                 spatial_lr_scale=sc["spatial_lr_scale"])
        bg = torch.zeros(3)
        view = engine.ViewArgs(H, W, cam.tanfovx, cam.tanfovy, 1.0, deg, cam.world_view_transform.t().contiguous().to(dev),
                               cam.projection_matrix.t().contiguous().to(dev), bg.to(dev))
        color, depth, alpha, radii, state = engine.render_forward(scene, view)
        act = state.geom["dbg_activated"].cpu()
    finally:
        engine.config.debug_activated = False
    feat = torch.cat([torch.cat((sc[k]["features_dc"], sc[k]["features_rest"]), 1) for k in ("static", "dynamic")], 0)
    orc = so.rasterize(act[:, 0:3].contiguous(), None, feat, None, act[:, 10:11].contiguous(), act[:, 3:6].contiguous(),
                       act[:, 6:10].contiguous(), cam.world_view_transform.t().contiguous(), helpers.oracle_settings(cam, bg, deg))
    D = int(state.num_rendered[0].item())
    assert torch.equal(radii.cpu(), orc.radii), "radii"
    assert D == orc.bn.keys.numel(), "duplicate count"
    assert torch.equal(state.extras["keys_sorted"][:D].cpu(), orc.bn.keys), "sorted keys"
    assert torch.equal(state.vals_sorted[:D].cpu(), orc.bn.vals), "sorted order"
    assert torch.equal(state.ranges.cpu(), orc.bn.ranges), "tile ranges"
    for name, a, b in (("color", color, orc.color), ("depth", depth, orc.depth), ("alpha", alpha, orc.alpha), ("final_T", state.final_T, orc.bl.final_T)):
        err = (a.cpu() - b).abs().max().item()
        assert err <= IMG_TOL, f"{name}: max-abs {err:.3e}"
    return D


def test_baseline_config_1_exactly():
    """BASELINE.json configs[0]: 10K Gaussians (50 % dynamic), 256x256, 8 frames - two of the frames, forward and all gradients."""
    N, H, W, T, _ = synthetic.CONFIGS["c1_cpu"]
    assert (N, H, W, T) == (10000, 256, 256, 8)
    sc = synthetic.make_scene(N, H, W, T, seed=0)
    for frame in (0, 5):
        cam = synthetic.make_camera(frame, 8, H, W, T)
        _fused_forward_on_own_activations(sc, cam, H, W)
        img_err, mism, errs, elem, D = _fused_vs_chain(sc, cam, H, W, seed=frame)
        assert img_err <= 2e-3 and mism <= 2e-3    # vs the CPU's activations: a stray 1/255 threshold may flip (strict check above)
        for k, e in errs.items():
            assert e <= GRAD_TOL, f"frame {frame} grad {k}: {e:.3e}"
        for k, res in elem.items():
            assert res[0], f"frame {frame} {k} element-wise: {res[1]:.2f} x the bound"


def test_density_matched_window_of_the_bench_workload():
    """The sample bench.py's CPU arm times: config 4's Gaussian density per tile on a 256x256 window, T = 100."""
    Nf, Hf, Wf, T, _ = synthetic.CONFIGS["c4_iphone"]
    tiles_f = ((Hf + 15) // 16) * ((Wf + 15) // 16)
    H = W = 256
    N = int(round(Nf * 256 / tiles_f))
    assert N == 62745
    sc = synthetic.make_scene(N, H, W, T, seed=0)
    cam = synthetic.make_camera(0, 8, H, W, T)
    D = _fused_forward_on_own_activations(sc, cam, H, W)
    assert D / 256 > 600, f"window is not as dense as the workload ({D / 256:.0f} entries per tile)"
    img_err, mism, errs, elem, D = _fused_vs_chain(sc, cam, H, W, truth64=True)
    assert img_err <= 2e-3 and mism <= 2e-3        # vs the CPU's activations: a stray 1/255 threshold may flip (strict check above)
    for k, e in errs.items():
        assert e <= GRAD_TOL, f"grad {k}: {e:.3e}"
    # 700+ list entries per tile and ~300 Gaussians per table row: the float32 oracle itself misses its float64 twin by up to
    # 7 x the element-wise bound here (cancellation), so the float64 chain is the yardstick (elementwise_vs_truth)
    for k, (ok, r_cu, r_32) in elem.items():
        assert ok, f"{k} element-wise vs float64: {r_cu:.2f} x the bound (float32 oracle: {r_32:.2f} x)"


def _adversarial(case, n, H, W, seed):
    """Activated tensors built to stress the band-solved sub-tile masks."""
    g = torch.Generator().manual_seed(seed)
    cam = synthetic.make_camera(1, 4, H, W, 4)
    f = W / (2.0 * cam.tanfovx)                                      # pixels per unit of x / z
    V = cam.world_view_transform.t()                                 # math V (row-major)
    z = 2.0 + 4.0 * torch.rand(n, generator=g)
    radius_px = {"tiny": 0.5, "large": 40.0, "huge": 200.0, "needle": 25.0, "mixed": 12.0}[case]
    # centres: inside the image and up to two radii outside of it
    margin = 2.0 * radius_px
    px = -margin + (W + 2 * margin) * torch.rand(n, generator=g)
    py = -margin + (H + 2 * margin) * torch.rand(n, generator=g)
    xv = (px - (W - 1) / 2.0) / f * z
    yv = (py - (H - 1) / 2.0) / f * z
    pv = torch.stack([xv, yv, z, torch.ones(n)], 1)
    xyz = (torch.linalg.inv(V) @ pv.t()).t()[:, :3].contiguous()
    sigma = radius_px / 3.0 * z / f                                  # world-space sigma for that screen radius
    scl = sigma.unsqueeze(1) * torch.exp(0.2 * torch.randn(n, 3, generator=g))
    if case == "needle":
        scl[:, 1:] = scl[:, :1] / 100.0                              # 100:1 anisotropy
    if case == "mixed":
        scl = scl * torch.exp(1.5 * torch.randn(n, 1, generator=g))
    rot = torch.randn(n, 4, generator=g)
    rot = rot / rot.norm(dim=1, keepdim=True)
    logit = torch.where(torch.rand(n, generator=g) < 0.5, torch.full((n,), -5.5), torch.full((n,), 6.0))
    if case == "mixed":
        logit = 3.0 * torch.randn(n, generator=g)
    op = torch.sigmoid(logit).unsqueeze(1)
    feat = torch.cat([torch.randn(n, 1, 3, generator=g), 0.1 * torch.randn(n, 15, 3, generator=g)], 1)
    return (xyz, op, scl, rot, feat), cam


@pytest.mark.parametrize("case,n,mod", [("tiny", 3000, 1.0), ("large", 300, 1.0), ("huge", 60, 1.0), ("needle", 500, 1.0),
                                        ("mixed", 1500, 0.3), ("mixed", 400, 3.0), ("needle", 300, 3.0), ("large", 300, 0.3)])
def test_sub_tile_masks_under_adversarial_footprints(case, n, mod):
    H, W = 112, 176
    acts, cam = _adversarial(case, n, H, W, seed=len(case) * 1000 + n)
    bg = torch.tensor([0.1, 0.2, 0.3])
    gen = torch.Generator().manual_seed(3)
    up = (torch.randn(3, H, W, generator=gen), 0.3 * torch.randn(1, H, W, generator=gen), 0.2 * torch.randn(1, H, W, generator=gen))
    xyz, op, scl, rot, feat = [t.detach().clone().requires_grad_(True) for t in acts]
    vm = cam.world_view_transform.t().contiguous().requires_grad_(True)
    m2 = torch.zeros(n, 3, requires_grad=True)
    orc = so.rasterize(xyz, m2, feat, None, op, scl, rot, vm, helpers.oracle_settings(cam, bg, 3, mod))
    ((orc.color * up[0]).sum() + (orc.depth * up[1]).sum() + (orc.alpha * up[2]).sum()).backward()
    assert int((orc.radii > 0).sum()) > n // 4
    out, g = _boundary(acts, cam.world_view_transform.t().contiguous(), cam.projection_matrix.t().contiguous(),
                       (cam.tanfovx, cam.tanfovy), H, W, bg, 3, up, mod)
    assert torch.equal(out[4].cpu(), orc.radii), "radii differ"
    # 100:1 needles have conics whose float32 evaluation itself is off by far more than 1e-4 (power is a difference of
    # terms ~1e5): there the bar is the float64 oracle, with the float32 oracle's own distance to it as the yardstick
    d64 = lambda t: t.detach().double()
    st64 = so.Settings(H, W, cam.tanfovx, cam.tanfovy, d64(bg), mod, d64(cam.projection_matrix.t().contiguous()), 3)
    o64 = so.rasterize(d64(xyz), torch.zeros(n, 3).double(), d64(feat), None, d64(op), d64(scl), d64(rot), d64(vm), st64)
    for name, a, b, b64 in (("color", out[0], orc.color, o64.color), ("depth", out[1], orc.depth, o64.depth), ("alpha", out[3], orc.alpha, o64.alpha)):
        err = (a.cpu() - b).abs().max().item()
        noise = (b.double() - b64).abs().max().item()
        err64 = (a.cpu().double() - b64).abs().max().item()
        assert err <= IMG_TOL or err64 <= 1.5 * noise + IMG_TOL, \
            f"{case} x{mod} {name}: max-abs {err:.3e} vs float32 oracle, {err64:.3e} vs float64 (float32 oracle itself: {noise:.3e})"
    ref = {"means3D": xyz.grad, "means2D": m2.grad, "shs": feat.grad, "opacities": op.grad, "scales": scl.grad, "rotations": rot.grad,
           "viewmatrix": vm.grad}
    l64 = {k: d64(t).requires_grad_(True) for k, t in (("means3D", xyz), ("opacities", op), ("scales", scl), ("rotations", rot), ("shs", feat), ("viewmatrix", vm))}
    l64["means2D"] = torch.zeros(n, 3, dtype=torch.float64, requires_grad=True)
    o64g = so.rasterize(l64["means3D"], l64["means2D"], l64["shs"], None, l64["opacities"], l64["scales"], l64["rotations"], l64["viewmatrix"], st64)
    ((o64g.color * up[0].double()).sum() + (o64g.depth * up[1].double()).sum() + (o64g.alpha * up[2].double()).sum()).backward()
    for k, r in ref.items():
        ok, e, noise = normwise_vs_truth(g[k], r, l64[k].grad)
        assert ok, f"{case} x{mod} grad {k}: {e:.3e} (float32 oracle vs float64: {noise:.3e})"
    # dL/dV element-wise: the yardstick is the float32 oracle's error, which has one fixed summation order.  The default
    # backward adds its partials with float atomics in an order that changes from run to run, and for 100:1 needles at x3
    # (heavy cancellation) that alone moves dL/dV between 1.0 and 2.6 x the bound on identical inputs.  The deterministic
    # backward fixes the order, so the element-wise bar is applied to it.
    engine.config.deterministic = True
    _, gd = _boundary(acts, cam.world_view_transform.t().contiguous(), cam.projection_matrix.t().contiguous(),
                      (cam.tanfovx, cam.tanfovy), H, W, bg, 3, up, mod)
    ok, r_cu, r_32 = elementwise_vs_truth(gd["viewmatrix"], ref["viewmatrix"], l64["viewmatrix"].grad)
    assert ok, f"{case} x{mod} dL/dV element-wise vs float64: {r_cu:.2f} x the bound (float32 oracle: {r_32:.2f} x)"

def _mask_coverage(acts, cam, H, W, mod, deg=3):
    """Directly checks the conservative sub-tile masks (blend.cu::rdg_sub_mask) on the region lists the forward pass wrote:
    every (list entry, pixel) pair that the per-pixel rule accepts with a 2 % margin (alpha >= 1.02 / 255, power <= 0,
    evaluated in float64 from the packed float32 records) must lie in a sub-tile of the entry's mask.  Returns the number
    of accepted pairs and the fraction of mask bits without any accepted pixel (tightness; informational)."""
    xyz, op, scl, rot, feat = [t.cuda() for t in acts]
    scene = engine.SceneArgs(st=engine.SetArgs(xyz=xyz, scaling=scl, rotation=rot, opacity=op, sh_dc=feat, sh_rest=feat,
                                               sh_dc_stride=48, sh_rest_stride=48, sh_rest_offset=3), raw=False)
    view = engine.ViewArgs(H, W, cam.tanfovx, cam.tanfovy, mod, deg, cam.world_view_transform.t().contiguous().cuda(),
                           cam.projection_matrix.t().contiguous().cuda(), torch.zeros(3).cuda())
    _, _, _, _, st = engine.render_forward(scene, view)
    p0, p1 = st.geom["p0"].double(), st.geom["p1"].double()
    ranges, vals = st.ranges.cpu().long(), st.vals_sorted.long()
    rid, rmask, rcount = st.extras["region_ids"].long(), st.extras["region_masks"].long(), st.extras["region_count"].cpu().long()
    stride = st.d_cap
    gx = (W + 15) // 16
    yy, xx = torch.meshgrid(torch.arange(16, device="cuda"), torch.arange(16, device="cuda"), indexing="ij")
    sub_of_pixel = ((yy // 4) * 4 + xx // 4).reshape(1, -1)          # [1,256]
    accepted = covered_bits = empty_bits = 0
    N = xyz.shape[0]
    for t in range(ranges.shape[0]):
        lo, hi = int(ranges[t, 0]), int(ranges[t, 1])
        if hi <= lo:
            continue
        ids = vals[lo:hi]
        mask16 = torch.zeros(N, dtype=torch.long, device="cuda")
        for r in range(2):
            c = int(rcount[2 * t + r])
            sl = slice(r * stride + lo, r * stride + lo + c)
            mask16[rid[sl] & 0x7fffffff] |= rmask[sl] << (8 * r)
        m = mask16[ids].unsqueeze(1)                                 # [n,1]
        tx, ty = t % gx, t // gx
        dx = p0[ids, 0:1] - (tx * 16 + xx.reshape(1, -1)).double()
        dy = p0[ids, 1:2] - (ty * 16 + yy.reshape(1, -1)).double()
        power = -0.5 * (p0[ids, 2:3] * dx * dx + p1[ids, 0:1] * dy * dy) - p0[ids, 3:4] * dx * dy
        alpha = p1[ids, 1:2] * torch.exp(power)
        inside = ((tx * 16 + xx.reshape(1, -1)) < W) & ((ty * 16 + yy.reshape(1, -1)) < H)
        acc = (power <= 0) & (alpha >= 1.02 / 255.0) & inside
        in_mask = ((m >> sub_of_pixel) & 1).bool()
        bad = acc & ~in_mask
        assert not bool(bad.any()), (f"tile {t}: {int(bad.sum())} accepted (entry, pixel) pairs outside the entry's sub-tile mask; "
                                     f"first entry id {int(ids[bad.any(1)][0])}")
        accepted += int(acc.sum())
        for s_ in range(16):
            bit = ((m[:, 0] >> s_) & 1).bool()
            has = (acc & (sub_of_pixel == s_)).any(1)
            covered_bits += int(bit.sum())
            empty_bits += int((bit & ~has).sum())
    return accepted, empty_bits / max(covered_bits, 1)


@pytest.mark.parametrize("case,n,mod", [("tiny", 3000, 1.0), ("large", 300, 1.0), ("huge", 60, 1.0), ("needle", 500, 1.0),
                                        ("needle", 300, 3.0), ("mixed", 1500, 0.3), ("mixed", 400, 3.0), ("plain", 6000, 1.0)])
def test_sub_tile_masks_cover_every_accepted_pixel(case, n, mod):
    H, W = 112, 176
    if case == "plain":
        sc, cam = helpers.small_scene(n, H, W, 4, seed=8, radius_px=5.0)
        acts = [a.detach() for a in helpers.activated_concat(sc, cam)]
    else:
        acts, cam = _adversarial(case, n, H, W, seed=len(case) * 1000 + n)
    accepted, slack = _mask_coverage(acts, cam, H, W, mod)
    assert accepted > 1000
    print(f"{case} x{mod}: {accepted} accepted pairs, {100 * slack:.1f} % of the mask bits have no accepted pixel")
