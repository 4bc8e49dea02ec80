"""Every backward kernel element-wise against float64, each one in isolation on its own inputs.

End-to-end gradient checks compare whole chains, so the CPU and the kernel may take a different side of an ambiguous
decision (an exp() ulp flips a radius or a 1/255 threshold) and float atomics reorder the sums; the large per-Gaussian
tensors are therefore only held norm-wise there, which lets a kernel get every small entry wrong.  Here:
  * rdg_blend_bwd / rdg_blend_bwd_deterministic run on the packed float32 records and the tile lists the forward kernel
    wrote; the float64 oracle blends exactly those records.  Pixels where any decision of the float64 replay lies within
    a small margin of its threshold get a zero upstream gradient in both runs (the gradients are linear in it), so no
    decision that float32 and float64 may take differently remains.  Ragged image sizes (every H % 16, W % 16 class the
    workloads have, 1920x1080 and 960x540 included) put the bottom / right partial tiles under test.
  * rdg_preprocess_bwd runs on an acc the test chooses; the float64 reference is autograd of the oracle chain
    (deform_oracle.assemble -> splat_oracle.preprocess) with acc's columns as grad_outputs, over every kernel instance:
    both input paths, SH degrees 0..3, colours given, scale modifier, pose-gradient switches, basis counts, empty models,
    chunk tails and the launch tunables.
  * rdg_sh_grad_views / rdg_sh_adam_views against sh_grad_from_factors (+ a float64 Adam step).
Bar, per element: |a - b64| <= 1e-3 |b64| + 1e-5 max|b64|; where the float32 oracle itself misses that bar on the same
inputs, 1.5 x the float32 oracle's own ratio.  test_elementwise_bar_rejects_what_the_normwise_bar_lets_through (CPU)
shows what the element-wise bar catches that the norm-wise one does not."""
import ctypes as C
import math

import pytest
import torch

import helpers
from oracle import deform_oracle as do
from oracle import splat_oracle as so
from rodygs_b200 import _lib, engine, synthetic
from rodygs_b200._lib import RdgBins, RdgImage, RdgSceneGrad, check, ptr

RTOL, FLOOR = 1e-3, 1e-5
ACC_COLS = ("dpx", "dpy", "dA", "dB", "dC", "dop", "dr", "dg", "db", "ddepth")
TUNABLES = {"pre_grid_cap": 0, "dtable_v1": 0, "diff_smem": 1, "l2_prefetch": 0, "sm_reserve": 0, "deterministic": 0}


def _ratio(got, ref64):
    got, ref64 = got.double().cpu(), ref64.double().cpu()
    bound = (RTOL * ref64.abs() + FLOOR * ref64.abs().max()).clamp_min(1e-300)
    return ((got - ref64).abs() / bound).max().item()


def _check(name, got, ref64, ref32=None, table=None):
    """Element-wise bar; the 1.5 x float32-oracle fallback only where the float32 oracle misses the bar itself."""
    r_cu = _ratio(got, ref64)
    r_32 = _ratio(ref32, ref64) if ref32 is not None else float("nan")
    ok = r_cu <= 1.0 or (r_32 > 1.0 and r_cu <= 1.5 * r_32)
    if table is not None:
        table.append(f"{name}: {r_cu:.3f}" + ("" if ref32 is None else f" (f32 oracle {r_32:.3f})"))
    assert ok, f"{name}: element-wise {r_cu:.3f} x (1e-3 |b| + 1e-5 max|b|) vs float64 (float32 oracle: {r_32:.3f} x)"


@pytest.fixture(autouse=True)
def _reset():
    yield
    for name, v in TUNABLES.items():
        _lib.set_tunable(name, v)
    engine.config.binning = "tiles"
    engine.config.deterministic = False
    engine.config.debug_keep_unsorted = False


# ------------------------------------------------------------------------------------------------------------- scenes --

def _cam_view(cam, deg=3, mod=1.0, bg=None, cov=True, sh=True):
    bg = torch.tensor([0.1, 0.2, 0.3]) if bg is None else bg
    return engine.ViewArgs(cam.height, cam.width, cam.tanfovx, cam.tanfovy, mod, deg,
                           cam.world_view_transform.t().contiguous().cuda(), cam.projection_matrix.t().contiguous().cuda(),
                           bg.cuda(), cov, sh)


def _boundary_scene(acts, colors=None):
    xyz, op, scl, rot, feat = [t.detach().contiguous().cuda() for t in acts]
    return engine.SceneArgs(st=engine.SetArgs(xyz=xyz, scaling=scl, rotation=rot, opacity=op, sh_dc=feat, sh_rest=feat,
                                              sh_dc_stride=48, sh_rest_stride=48, sh_rest_offset=3), raw=False,
                            colors_precomp=None if colors is None else colors.contiguous().cuda())


def _placed(cam, px, py, radius_px, seed):
    """Activated Gaussians at given pixel centres with ~radius_px screen radius (depth 2..6)."""
    g = torch.Generator().manual_seed(seed)
    n = px.shape[0]
    H, W = cam.height, cam.width
    f = W / (2.0 * cam.tanfovx)
    V = cam.world_view_transform
    z = 2.0 + 4.0 * torch.rand(n, generator=g)
    pv = torch.stack([(px - (W - 1) / 2.0) / f * z, (py - (H - 1) / 2.0) / f * z, z, torch.ones(n)], 1)
    xyz = (torch.linalg.inv(V) @ pv.t()).t()[:, :3].contiguous()
    sigma = radius_px / 3.0 * z / f
    scl = sigma.unsqueeze(1) * torch.exp(0.4 * torch.randn(n, 3, generator=g))
    rot = torch.randn(n, 4, generator=g)
    rot = rot / rot.norm(dim=1, keepdim=True)
    op = torch.sigmoid(-0.5 + 1.5 * torch.randn(n, 1, generator=g))
    feat = torch.cat([torch.randn(n, 1, 3, generator=g), 0.1 * torch.randn(n, 15, 3, generator=g)], 1)
    return xyz, op, scl, rot, feat


def _edge_bands(H, W, n, seed):
    """Gaussians only in bands around the last tile row and the last tile column of a full-size camera."""
    g = torch.Generator().manual_seed(seed)
    cam = synthetic.make_camera(1, 8, H, W, 4)
    row0, col0 = 16 * ((H - 1) // 16), 16 * ((W - 1) // 16)
    h = n // 2
    px = torch.cat([(W + 16) * torch.rand(h, generator=g) - 8, col0 - 12 + (W + 20 - col0) * torch.rand(n - h, generator=g)])
    py = torch.cat([row0 - 12 + (H + 20 - row0) * torch.rand(h, generator=g), (H + 16) * torch.rand(n - h, generator=g) - 8])
    return _placed(cam, px, py, 6.0, seed), cam


# -------------------------------------------------------------------------------------------- part 1: blend backward --

def _blend_bwd(state, up, det):
    """rdg_blend_bwd / rdg_blend_bwd_deterministic on the forward's own records and lists -> acc [N,12] (CPU)."""
    lib = _lib.load()
    n = state.n
    acc = torch.zeros(max(n, 1), engine.NACC, device="cuda")
    gm_s, vw_s = engine._geom_struct(state.geom), engine._view_struct(state.view)
    bins = RdgBins()
    bins.vals_sorted, bins.ranges, bins.num_rendered = ptr(state.vals_sorted), ptr(state.ranges), ptr(state.num_rendered)
    bins.region_ids, bins.region_masks = ptr(state.extras["region_ids"]), ptr(state.extras["region_masks"])
    bins.region_count, bins.region_stride = ptr(state.extras["region_count"]), state.d_cap
    img = RdgImage()
    img.final_T, img.n_contrib = ptr(state.final_T), ptr(state.n_contrib)
    gc, gd, ga = [t.contiguous().cuda() for t in up]
    stream = _lib.stream_ptr()
    if det:
        nb = int(lib.rdg_blend_bwd_deterministic_scratch_bytes(n))
        scratch = torch.empty(max(nb, 8), dtype=torch.uint8, device="cuda")
        check(lib.rdg_blend_bwd_deterministic(n, C.byref(gm_s), C.byref(bins), C.byref(vw_s), C.byref(img), ptr(gc), ptr(gd),
                                              ptr(ga), ptr(acc), ptr(scratch), nb, stream))
    else:
        check(lib.rdg_blend_bwd(n, C.byref(gm_s), C.byref(bins), C.byref(vw_s), C.byref(img), ptr(gc), ptr(gd), ptr(ga),
                                ptr(acc), stream))
    return acc.cpu()


def _records(state, dt):
    """The packed records the forward wrote, as leaves of dtype dt (xy in pixels, conic (A, B, C), opacity, rgb, depth)."""
    p0, p1, p2 = [state.geom[k].cpu().to(dt) for k in ("p0", "p1", "p2")]
    return {"xy": p0[:, :2].clone(), "conic": torch.stack([p0[:, 2], p0[:, 3], p1[:, 0]], 1),
            "opacity": p1[:, 1].clone(), "rgb": torch.stack([p1[:, 2], p1[:, 3], p2[:, 0]], 1), "depth": p2[:, 1].clone()}


def _oracle_acc(rec, vals, ranges, bg, H, W, up):
    """splat_oracle.blend over the records + autograd -> (acc [N,10] in the kernel's column order, Blended)."""
    leaves = {k: v.clone().requires_grad_(True) for k, v in rec.items()}
    pp = so.Preprocessed(idx=None, visible=None, radii=None, tiles_touched=None, rect_min=None, rect_max=None,
                         xy=leaves["xy"], depth=leaves["depth"], conic=leaves["conic"], opacity=leaves["opacity"],
                         rgb=leaves["rgb"], cov2d=None)
    bn = so.Binned(None, None, None, None, local=vals, ranges=ranges, point_offsets=None)
    dt = rec["xy"].dtype
    bl = so.blend(pp, bn, bg.to(dt), H, W)
    loss = (bl.color * up[0].to(dt)).sum() + (bl.depth * up[1].to(dt)).sum() + (bl.alpha * up[2].to(dt)).sum()
    if loss.requires_grad:
        loss.backward()
    g = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in leaves.items()}
    acc = torch.cat([g["xy"], g["conic"], g["opacity"].unsqueeze(1), g["rgb"], g["depth"].unsqueeze(1)], 1)
    return acc, bl


@torch.no_grad()
def _replay(rec, state, H, W, margin=1e-6, t_margin=2e-4):
    """float64 replay of every (entry, pixel) decision of the kernel's lists.  Returns (flagged [H,W]: a decision within the
    margin of its threshold - power <= 0, alpha >= 1/255, the 0.99 clamp, T < 1e-4 - at an entry the pixel still reaches,
    n_contrib [H,W] in the kernel's convention: the REGION-list position the pixel stopped at, or the region's length).
    The margin of the power / alpha tests scales with the magnitude of the terms of the float32 quadratic form."""
    gx, gy = (W + 15) // 16, (H + 15) // 16
    D = int(state.num_rendered[0])
    vals = state.vals_sorted[:D].cpu().long()
    ranges = state.ranges.cpu().long()
    rid = state.extras["region_ids"].cpu().long() & 0x7fffffff
    rcount = state.extras["region_count"].cpu().long()
    stride = state.d_cap
    flag = torch.zeros(gy * 16, gx * 16, dtype=torch.bool)
    ncon = torch.zeros(gy * 16, gx * 16, dtype=torch.long)
    yy, xx = torch.meshgrid(torch.arange(16), torch.arange(16), indexing="ij")
    yy, xx = yy.reshape(1, -1), xx.reshape(1, -1)
    posmap = torch.full((state.n,), -1, dtype=torch.long)
    xy, con, op = rec["xy"], rec["conic"], rec["opacity"]
    for t in range(gx * gy):
        lo, hi = int(ranges[t, 0]), int(ranges[t, 1])
        ty, tx = t // gx, t % gx
        if hi <= lo:
            continue
        g = vals[lo:hi]
        dx = xy[g, 0:1] - (tx * 16 + xx).double()
        dy = xy[g, 1:2] - (ty * 16 + yy).double()
        ta, tb, tc = 0.5 * con[g, 0:1] * dx * dx, con[g, 1:2] * dx * dy, 0.5 * con[g, 2:3] * dy * dy
        power = -(ta + tc) - tb
        m = margin * (ta.abs() + tb.abs() + tc.abs() + 1.0)
        a = op[g].reshape(-1, 1) * torch.exp(power)
        valid = (power <= 0) & (a >= so.ALPHA_MIN)
        a_eff = torch.where(valid, a.clamp_max(so.ALPHA_MAX), torch.zeros_like(a))
        T_incl = torch.cumprod(1.0 - a_eff, 0)
        T_excl = torch.cat([torch.ones(1, 256, dtype=torch.float64), T_incl[:-1]], 0)
        reach = T_excl >= so.T_STOP * (1.0 - t_margin)
        la = torch.log(a * 255.0)
        near = (((power.abs() <= m) & (la >= -(m + margin)))
                | (la.abs() <= m + margin)
                | (torch.log(a / so.ALPHA_MAX).abs() <= m + margin)
                | (valid & (torch.log(T_incl / so.T_STOP).abs() <= t_margin)))
        flag[ty * 16:ty * 16 + 16, tx * 16:tx * 16 + 16] = (near & reach).any(0).reshape(16, 16)
        stop = valid & (T_incl < so.T_STOP)
        stopped = stop.any(0)
        first = torch.where(stopped, stop.to(torch.int8).argmax(0), torch.full((256,), hi - lo, dtype=torch.long))
        posmap[g] = torch.arange(hi - lo)
        exp_nc = torch.zeros(256, dtype=torch.long)
        for r in range(2):
            cnt = int(rcount[2 * t + r])
            rpos = posmap[rid[r * stride + lo:r * stride + lo + cnt]]
            assert bool((rpos >= 0).all()) and bool((rpos[1:] > rpos[:-1]).all()), f"tile {t} region {r}: not a sub-list"
            sel = (yy[0] // 8) == r
            exp_nc[sel] = torch.where(stopped[sel], torch.searchsorted(rpos, first[sel]), torch.full_like(first[sel], cnt))
        posmap[g] = -1
        ncon[ty * 16:ty * 16 + 16, tx * 16:tx * 16 + 16] = exp_nc.reshape(16, 16)
    return flag[:H, :W], ncon[:H, :W]


def _blend_case(scene, view, seed, max_flagged=0.01):
    H, W = int(view.height), int(view.width)
    color, depth, alpha, radii, state = engine.render_forward(scene, view)
    D = int(state.num_rendered[0])
    assert D > 0
    rec64, rec32 = _records(state, torch.float64), _records(state, torch.float32)
    flag, ncon = _replay(rec64, state, H, W)
    frac = flag.float().mean().item()
    g = torch.Generator().manual_seed(seed)
    keep = (~flag).float()
    up = tuple(s * torch.randn(c, H, W, generator=g) * keep for s, c in ((1.0, 3), (0.3, 1), (0.2, 1)))
    vals, ranges = state.vals_sorted[:D].cpu().long(), state.ranges.cpu()
    bg = state.view.bg.cpu()
    acc64, bl64 = _oracle_acc(rec64, vals, ranges, bg, H, W, up)
    acc32, bl32 = _oracle_acc(rec32, vals, ranges, bg, H, W, up)
    lines = [f"{H}x{W}: {D / max(1, ((H + 15) // 16) * ((W + 15) // 16)):.0f} entries/tile, flagged pixels {100 * frac:.3f} %"]
    # the forward on the unflagged pixels: n_contrib bit-exact, images at float32 resolution
    ok = ~flag
    nc = state.n_contrib.cpu().long()
    bad = ok & (nc != ncon)
    assert not bool(bad.any()), f"n_contrib differs at {int(bad.sum())} unflagged pixels, first {bad.nonzero()[0].tolist()}"
    # (100:1 needles: power is a difference of terms ~1e4, so float32 itself is off by more than 2e-6 there - the float32
    # oracle on the same records is the yardstick where it misses the bar, as for the gradients)
    for name, a, b, b32 in (("color", color, bl64.color, bl32.color), ("depth", depth, bl64.depth, bl32.depth),
                            ("alpha", alpha, bl64.alpha, bl32.alpha), ("final_T", state.final_T, bl64.final_T, bl32.final_T)):
        a, b, b32 = [t.detach().cpu().double().reshape(-1, H, W) for t in (a, b, b32)]
        rel = lambda x: ((x - b).abs() / (1.0 + b.abs()))[:, ok].max().item() if bool(ok.any()) else 0.0
        err, err32 = rel(a), rel(b32)
        assert err <= 2e-6 or (err32 > 2e-6 and err <= 1.5 * err32), \
            f"{name}: {err:.3e} relative to 1 + |b64| on unflagged pixels (float32 oracle: {err32:.3e})"
    assert frac < max_flagged, f"{100 * frac:.2f} % of the pixels have an ambiguous decision"
    for det in (False, True):
        acc = _blend_bwd(state, up, det)[:, :10]
        tag = "deterministic" if det else "atomics"
        row = []
        for c, name in enumerate(ACC_COLS):
            _check(f"{tag} {name}", acc[:, c], acc64[:, c], acc32[:, c], row)
        lines.append(f"  {tag}: " + "; ".join(r.split(" ", 1)[1] for r in row))
        assert torch.equal(acc[state.n:], torch.zeros_like(acc[state.n:]))
    print("\n".join(lines))
    return state, acc64


RAGGED = [(88, 136, 2500, 5.0), (76, 150, 2500, 5.0), (97, 131, 3000, 5.0), (7, 45, 200, 4.0), (9, 16, 80, 4.0),
          (200, 17, 600, 4.0), (8, 300, 600, 4.0), (16, 16, 120, 4.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,n,radius", RAGGED)
def test_blend_bwd_elementwise_on_ragged_images(H, W, n, radius):
    sc, cam = helpers.small_scene(n, H, W, 6, seed=H * 1000 + W, radius_px=radius)
    acts = helpers.activated_concat(sc, cam)
    _blend_case(_boundary_scene(acts), _cam_view(cam), seed=H + W)


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,n", [(1080, 1920, 4000), (540, 960, 2500)])
def test_blend_bwd_elementwise_at_production_geometries(H, W, n):
    """1080 % 16 = 8: region 1 of every bottom tile lies entirely outside the image; 540 % 16 = 12: it has 4 of 8 rows."""
    acts, cam = _edge_bands(H, W, n, seed=H)
    _blend_case(_boundary_scene(acts), _cam_view(cam), seed=W)


@pytest.mark.gpu
def test_blend_bwd_elementwise_dense():
    """Hundreds of list entries per tile: long region lists, several staging rounds, pixels that saturate (T < 1e-4)."""
    H, W = 88, 136
    sc, cam = helpers.small_scene(30000, H, W, 6, seed=77, radius_px=7.0)
    acts = helpers.activated_concat(sc, cam)
    state, _ = _blend_case(_boundary_scene(acts), _cam_view(cam), seed=3)
    assert int(state.num_rendered[0]) / (6 * 9) > 300


@pytest.mark.gpu
@pytest.mark.parametrize("case,n,mod", [("needle", 300, 1.0), ("huge", 40, 1.0), ("large", 200, 3.0), ("tiny", 2000, 1.0)])
def test_blend_bwd_elementwise_adversarial_footprints(case, n, mod):
    """Needles (100:1) and splats of up to 200 px that cross the image edge, on a ragged 97x131 image."""
    from test_gpu_golden import _adversarial
    H, W = 97, 131
    acts, cam = _adversarial(case, n, H, W, seed=len(case) * 100 + n)
    _blend_case(_boundary_scene(acts), _cam_view(cam, mod=mod), seed=n, max_flagged=0.02)


# ------------------------------------------------------------------------------------- part 2: per-Gaussian backward --

def _split_scene(ns, nd, H, W, T, K, seed):
    """make_scene with exactly ns static and nd dynamic Gaussians."""
    m = max(ns, nd, 1)
    sc = synthetic.make_scene(2 * m, H, W, T, seed=seed, radius_px=5.0, num_basis=K)
    out = {"static": {k: v[:ns].contiguous() for k, v in sc["static"].items()},
           "dynamic": {k: v[:nd].contiguous() for k, v in sc["dynamic"].items()},
           "motion_coeff": sc["motion_coeff"][:nd].squeeze(1).contiguous(), "time_ind": sc["time_ind"][:nd].contiguous(),
           "table": sc["table"], "spatial_lr_scale": 1.3}
    return out


def _fused_args(sc, bt, dev="cuda"):
    def mk(d):
        if d["xyz"].shape[0] == 0:
            return None
        return engine.SetArgs(xyz=d["xyz"].to(dev), scaling=d["scaling"].to(dev), rotation=d["rotation"].to(dev),
                              opacity=d["opacity"].to(dev), sh_dc=d["features_dc"].to(dev), sh_rest=d["features_rest"].to(dev))
    nd = sc["dynamic"]["xyz"].shape[0]
    ti = sc["time_ind"].to(dev)
    order, offsets = engine.frame_csr(ti, sc["table"].shape[0]) if nd > 0 else (None, None)
    return engine.SceneArgs(st=mk(sc["static"]), dy=mk(sc["dynamic"]), raw=True, use_deform=nd > 0,
                            motion_coeff=sc["motion_coeff"].to(dev) if nd else None, time_ind=ti if nd else None,
                            basis_t=bt.contiguous().to(dev) if nd else None, table=sc["table"].to(dev) if nd else None,
                            spatial_lr_scale=sc["spatial_lr_scale"], frame_order=order, frame_offsets=offsets)


def _raw_rgb(xyz, feat, vm_glm, deg):
    """Unclamped SH colour + 0.5 (splat_oracle.preprocess step 9), float64."""
    V = vm_glm.t()
    cp = -(V[:3, :3].t() @ V[:3, 3])
    d = xyz - cp.reshape(1, 3)
    d = d / d.norm(dim=1, keepdim=True)
    return so.sh_to_rgb(deg, feat, d) + 0.5


PRE_CASES = [
    # path, deg, (ns, nd), K, T, extra
    ("boundary", 0, (1301, 0), 16, 6, {}), ("boundary", 1, (1301, 0), 16, 6, {}), ("boundary", 2, (1301, 0), 16, 6, {}),
    ("boundary", 3, (1301, 0), 16, 6, {}), ("boundary", 3, (1301, 0), 16, 6, {"acc": "real"}),
    ("boundary", 1, (1301, 0), 16, 6, {"acc": "real"}), ("boundary", 0, (1301, 0), 16, 6, {"colors": True}),
    ("boundary", 2, (1301, 0), 16, 6, {"mod": 0.7}), ("boundary", 3, (1301, 0), 16, 6, {"cov": False}),
    ("boundary", 3, (1301, 0), 16, 6, {"sh": False}), ("boundary", 3, (255, 0), 16, 6, {"l2_prefetch": 1}),
    ("fused", 0, (1301, 1302), 16, 6, {}), ("fused", 1, (1301, 1302), 16, 6, {}), ("fused", 2, (1301, 1302), 16, 6, {}),
    ("fused", 3, (1301, 1302), 16, 6, {}), ("fused", 3, (1301, 1302), 16, 6, {"acc": "real"}),
    ("fused", 1, (1301, 1302), 16, 6, {"acc": "real"}),
    ("fused", 3, (1301, 1302), 7, 6, {}), ("fused", 3, (1301, 1302), 7, 150, {}), ("fused", 2, (1301, 1302), 1, 6, {}),
    ("fused", 3, (1301, 1302), 1, 150, {}), ("fused", 3, (1301, 1302), 16, 150, {}),
    ("fused", 3, (0, 1301), 16, 6, {}), ("fused", 3, (1301, 0), 16, 6, {}), ("fused", 2, (1, 257), 16, 6, {}),
    ("fused", 3, (255, 256), 7, 6, {}),
    ("fused", 3, (1301, 1302), 16, 6, {"pre_grid_cap": 2}), ("fused", 3, (1301, 1302), 16, 6, {"dtable_v1": 1}),
    ("fused", 3, (1301, 1302), 7, 6, {"diff_smem": 0}), ("fused", 0, (1301, 1302), 16, 6, {"l2_prefetch": 1}),
    ("fused", 3, (3000, 3001), 16, 6, {"sm_reserve": 140}),
    ("fused", 3, (1301, 1302), 16, 6, {"cov": False}), ("fused", 2, (1301, 1302), 16, 6, {"sh": False, "mod": 1.4}),
]


def _case_id(c):
    path, deg, (ns, nd), K, T, ex = c
    return f"{path}-deg{deg}-{ns}+{nd}-K{K}-T{T}" + "".join(f"-{k}{v}" for k, v in ex.items())


@pytest.mark.gpu
@pytest.mark.parametrize("case", PRE_CASES, ids=[_case_id(c) for c in PRE_CASES])
def test_preprocess_bwd_elementwise_against_float64_autograd(case):
    path, deg, (ns, nd), K, T, ex = case
    H, W = 72, 100
    for name in TUNABLES:
        if name in ex:
            _lib.set_tunable(name, ex[name])
    mod, cov, shg = ex.get("mod", 1.0), ex.get("cov", True), ex.get("sh", True)
    seed = 1000 * deg + ns + 7 * nd + K + T
    sc = _split_scene(ns, nd, H, W, T, K, seed)
    cam = synthetic.make_camera(3, 8, H, W, T)
    gen = torch.Generator().manual_seed(seed)
    bt = sc["table"][cam.time_index] + 0.02 * torch.randn(K, 7, generator=gen)
    n = ns + nd
    f64 = torch.float64
    # ---- float64 leaves and the activated tensors the kernel sees ----
    def leaf(t):
        return t.detach().clone().to(f64).requires_grad_(True)
    colors = torch.rand(n, 3, generator=gen) if ex.get("colors") else None
    if path == "boundary":
        acts = helpers.activated_concat(synthetic.make_scene(2 * n, H, W, T, seed=seed), cam)
        acts = [a.detach()[:n].contiguous() for a in acts]
        scene = _boundary_scene(acts, colors)
        L = {k: leaf(v) for k, v in zip(("xyz", "opacity", "scaling", "rotation", "feat"), acts)}
        a64 = (L["xyz"], L["opacity"], L["scaling"], L["rotation"], L["feat"])
    else:
        scene = _fused_args(sc, bt)
        Ls = {k: leaf(v) for k, v in sc["static"].items()}
        Ld = {k: leaf(v) for k, v in sc["dynamic"].items()}
        coeff, table, basis = leaf(sc["motion_coeff"]), leaf(sc["table"]), leaf(bt)
        a64 = do.assemble(do.RawGaussians(**Ls), do.RawGaussians(**Ld), coeff, basis, table, sc["time_ind"].long(),
                          sc["spatial_lr_scale"], nd > 0)
    col64 = None if colors is None else leaf(colors)
    vm64 = leaf(cam.world_view_transform.t().contiguous())
    m2 = torch.zeros(n, 3, dtype=f64, requires_grad=True)
    view = _cam_view(cam, deg, mod, cov=cov, sh=shg)
    st64 = so.Settings(H, W, cam.tanfovx, cam.tanfovy, view.bg.cpu().to(f64), mod,
                       cam.projection_matrix.t().contiguous().to(f64), deg, False, False, cov, shg)
    pp = so.preprocess(a64[0], a64[2], a64[3], a64[1], None if colors is not None else a64[4], col64, vm64, st64, means2D=m2)
    # ---- the kernel's forward (radii, clamp flags) and the acc fed to the backward ----
    color, depth, alpha, radii, state = engine.render_forward(scene, view)
    if ex.get("acc") == "real":
        up = tuple(s * torch.randn(c, H, W, generator=gen) for s, c in ((1.0, 3), (0.3, 1), (0.2, 1)))
        acc = _blend_bwd(state, up, det=True)
    else:
        scales = torch.tensor([1.0, 1.0, 30.0, 30.0, 30.0, 1.0, 1.0, 1.0, 1.0, 0.3, 0.0, 0.0])
        acc = torch.randn(max(n, 1), 12, generator=gen) * scales
    acc = acc[:n].clone()
    # ambiguity removed through acc: rows whose visibility differs, channels whose float64 colour sits at the clamp
    r_cu = radii.cpu()
    vis64 = pp.radii > 0
    mismatch = (r_cu > 0) != vis64
    acc[~((r_cu > 0) & vis64)] = 0.0
    masked_ch = 0
    if colors is None:
        with torch.no_grad():
            raw = torch.zeros(n, 3, dtype=f64)
            raw[pp.idx] = _raw_rgb(a64[0].detach()[pp.idx], a64[4].detach()[pp.idx], vm64.detach(), deg)
        near = raw.abs() <= 1e-5
        acc[:, 6:9][near] = 0.0
        masked_ch = int(near[vis64].sum())
        cl = state.geom["clamped"].cpu().long()
        cl_bits = torch.stack([(cl >> c) & 1 for c in range(3)], 1).bool()
        vis_both = (r_cu > 0) & vis64
        disagree = vis_both.unsqueeze(1) & (cl_bits != (raw < 0)) & ~near
        assert not bool(disagree.any()), "clamp flags differ from the float64 colour away from the clamp"
    print(f"{_case_id(case)}: visibility mismatches {int(mismatch.sum())} / {n}, clamp-margin channels {masked_ch}")
    assert int(mismatch.sum()) <= max(2, n // 500) and masked_ch <= max(2, n // 500)
    # ---- float64 reference: autograd with acc's columns as grad_outputs ----
    A = acc.to(f64)[pp.idx]
    loss = ((pp.xy * A[:, 0:2]).sum() + (pp.conic * A[:, 2:5]).sum() + (pp.opacity * A[:, 5]).sum()
            + (pp.rgb * A[:, 6:9]).sum() + (pp.depth * A[:, 9]).sum())
    loss.backward()

    def g64(t):
        return t.grad if t.grad is not None else torch.zeros_like(t)
    # ---- the kernel ----
    dev = "cuda"
    f32 = dict(dtype=torch.float32, device=dev)
    acc_d = torch.zeros(max(n, 1), 12, **f32)
    acc_d[:n] = acc.to(dev)
    grads = engine.SceneGrads(means2D=torch.full((n, 3), 7.0, **f32), viewmatrix=torch.zeros(4, 4, **f32),
                              dcolor=torch.full((n, 3), 7.0, **f32))
    if path == "boundary":
        feat_g = torch.full((n, 16, 3), 7.0, **f32)
        grads.st = engine.SetGrads(xyz=torch.full((n, 3), 7.0, **f32), scaling=torch.full((n, 3), 7.0, **f32),
                                   rotation=torch.full((n, 4), 7.0, **f32), opacity=torch.full((n, 1), 7.0, **f32),
                                   sh_dc=feat_g if colors is None else None, sh_rest=feat_g if colors is None else None,
                                   sh_rest_offset=3)
        if colors is not None:
            grads.colors_precomp = torch.full((n, 3), 7.0, **f32)
    else:
        def sg(m):
            if m == 0:
                return engine.SetGrads()
            return engine.SetGrads(xyz=torch.full((m, 3), 7.0, **f32), scaling=torch.full((m, 3), 7.0, **f32),
                                   rotation=torch.full((m, 4), 7.0, **f32), opacity=torch.full((m, 1), 7.0, **f32),
                                   sh_dc=torch.full((m, 1, 3), 7.0, **f32), sh_rest=torch.full((m, 15, 3), 7.0, **f32))
        grads.st, grads.dy = sg(ns), sg(nd)
        if nd > 0:
            grads.motion_coeff = torch.full((nd, K), 7.0, **f32)
            grads.table = torch.zeros(T, K, 7, **f32)
            grads.basis_t = torch.zeros(K, 7, **f32)
            grads.g7_scratch = torch.empty(nd, 8, **f32)
    if ex.get("sm_reserve"):
        grads.sm_queue = torch.zeros(4, dtype=torch.int32, device=dev)
    g = RdgSceneGrad()
    g.st, g.dy = engine._setgrad_struct(grads.st), engine._setgrad_struct(grads.dy)
    g.colors_precomp, g.means2D, g.viewmatrix = ptr(grads.colors_precomp), ptr(grads.means2D), ptr(grads.viewmatrix)
    g.motion_coeff, g.table, g.basis_t = ptr(grads.motion_coeff), ptr(grads.table), ptr(grads.basis_t)
    g.g7_scratch, g.sm_queue, g.dcolor = ptr(grads.g7_scratch), ptr(grads.sm_queue), ptr(grads.dcolor)
    g.models = 0
    check(_lib.load().rdg_preprocess_bwd(C.byref(engine._scene_struct(state.scene)), C.byref(engine._view_struct(state.view)),
                                         C.byref(engine._geom_struct(state.geom)), ptr(acc_d), C.byref(g), _lib.stream_ptr()))
    torch.cuda.synchronize()
    if grads.sm_queue is not None:
        assert int(grads.sm_queue.abs().max()) == 0
    # ---- compare every output ----
    row = []
    pairs = [("means2D", grads.means2D, g64(m2)), ("viewmatrix", grads.viewmatrix, g64(vm64))]
    vis_rows = ((r_cu > 0) & vis64).unsqueeze(1).to(f64)
    rgb_mask = torch.ones(n, 3, dtype=f64) if colors is not None else (raw > 0).to(f64)
    pairs.append(("dcolor", grads.dcolor, acc.to(f64)[:, 6:9] * rgb_mask * vis_rows))
    if path == "boundary":
        pairs += [("means3D", grads.st.xyz, g64(L["xyz"])), ("scales", grads.st.scaling, g64(L["scaling"])),
                  ("rotations", grads.st.rotation, g64(L["rotation"])), ("opacities", grads.st.opacity, g64(L["opacity"]))]
        if colors is None:
            pairs.append(("shs", feat_g, g64(L["feat"])))
        else:
            pairs.append(("colors_precomp", grads.colors_precomp, g64(col64)))
    else:
        for tag, gs, Lx, m in (("static", grads.st, Ls, ns), ("dynamic", grads.dy, Ld, nd)):
            if m == 0:
                continue
            for k in ("xyz", "scaling", "rotation", "opacity", "features_dc", "features_rest"):
                key = {"features_dc": "sh_dc", "features_rest": "sh_rest"}.get(k, k)
                pairs.append((f"{tag}.{k}", getattr(gs, key), g64(Lx[k])))
            kk = (deg + 1) ** 2
            upper = gs.sh_rest[:, kk - 1:]
            assert torch.equal(upper, torch.zeros_like(upper)), f"{tag}: features_rest rows >= {kk} must get exactly 0"
        if nd > 0:
            pairs += [("motion_coeff", grads.motion_coeff, g64(coeff)), ("table", grads.table, g64(table)),
                      ("basis_t", grads.basis_t, g64(basis))]
    for name, got, ref in pairs:
        _check(name, got.reshape(ref.shape), ref, table=row)
    print("  " + "; ".join(row))


# ----------------------------------------------------------------------------- part 3: dL/dSH from per-view factors --

SGV_CASES = [(0, 1, 6, (1301, 1302), 16), (1, 3, 6, (255, 259), 16), (2, 5, 6, (1301, 1302), 7), (3, 16, 6, (1301, 1302), 16),
             (3, 5, 150, (1301, 1302), 16), (1, 16, 150, (0, 1301), 7), (3, 3, 6, (1301, 0), 16), (2, 1, 200, (3, 517), 1)]


def _sgv_inputs(deg, V, T, ns, nd, K, seed):
    H, W = 64, 96
    sc = _split_scene(ns, nd, H, W, T, K, seed)
    gen = torch.Generator().manual_seed(seed + 1)
    n = ns + nd
    cams = [synthetic.make_camera(v, 16, H, W, T) for v in range(V)]
    vms = torch.stack([c.world_view_transform.t().contiguous() for c in cams])
    bts = torch.stack([sc["table"][c.time_index] + 0.02 * torch.randn(K, 7, generator=gen) for c in cams]).contiguous()
    dcol = torch.randn(V, n, 3, generator=gen)
    dcol[torch.rand(V, n, generator=gen) < 0.3] = 0.0                     # not visible in that view
    dcol[torch.rand(V, n, 3, generator=gen) < 0.15] = 0.0                 # clamped channels
    scale = 1.0 / V
    # float64 reference: deformed means per view, directions from each view's camera centre
    f64 = torch.float64
    st = do.RawGaussians(**{k: v.to(f64) for k, v in sc["static"].items()})
    dy = do.RawGaussians(**{k: v.to(f64) for k, v in sc["dynamic"].items()})
    means, camps = [], []
    for v in range(V):
        xyz = do.assemble(st, dy, sc["motion_coeff"].to(f64), bts[v].to(f64), sc["table"].to(f64), sc["time_ind"].long(),
                          sc["spatial_lr_scale"], nd > 0)[0]
        Vm = vms[v].to(f64).t()
        means.append(xyz)
        camps.append(-(Vm[:3, :3].t() @ Vm[:3, 3]))
    ref = so.sh_grad_from_factors(deg, means, camps, [d.to(f64) for d in dcol]) * scale
    scene = _fused_args(sc, bts[0])
    return sc, scene, vms.cuda(), bts.cuda(), dcol.cuda(), scale, ref


@pytest.mark.gpu
@pytest.mark.parametrize("deg,V,T,sizes,K", SGV_CASES)
def test_sh_grad_views_elementwise_against_float64(deg, V, T, sizes, K):
    ns, nd = sizes
    sc, scene, vms, bts, dcol, scale, ref = _sgv_inputs(deg, V, T, ns, nd, K, seed=deg * 100 + V + T + K)
    f32 = dict(dtype=torch.float32, device="cuda")
    outs = {}
    structs = []
    for tag, m in (("static", ns), ("dynamic", nd)):
        gs = _lib.RdgSetGrad()
        if m:
            outs[tag] = (torch.full((m, 1, 3), 7.0, **f32), torch.full((m, 15, 3), 7.0, **f32))
            gs.sh_dc, gs.sh_rest = ptr(outs[tag][0]), ptr(outs[tag][1])
        structs.append(gs)
    check(_lib.load().rdg_sh_grad_views(C.byref(engine._scene_struct(scene)), deg, V, ptr(vms), ptr(bts), ptr(dcol), scale,
                                        C.byref(structs[0]), C.byref(structs[1]), None, _lib.stream_ptr()))
    K_sh = (deg + 1) ** 2
    row = []
    for tag, lo, m in (("static", 0, ns), ("dynamic", ns, nd)):
        if not m:
            continue
        dc, rest = outs[tag]
        _check(f"{tag}.dc", dc.cpu(), ref[lo:lo + m, :1], table=row)
        _check(f"{tag}.rest", rest.cpu(), ref[lo:lo + m, 1:], table=row)
        upper = rest[:, K_sh - 1:]
        assert torch.equal(upper, torch.zeros_like(upper)), f"{tag}: coefficients >= {K_sh} must be exactly 0"
    print(f"sh_grad_views deg {deg} V {V} T {T} {ns}+{nd} K {K}: " + "; ".join(row))


@pytest.mark.gpu
@pytest.mark.parametrize("deg", [2, 3])
def test_sh_grad_views_num_basis_below_16_with_the_table_in_shared_memory(deg):
    """Regression: the per-view deformation sums all 16 rows of B(t_v) with c_k = 0 beyond num_basis, but only num_basis rows
    were staged in shared memory, so 0 x a stale NaN / Inf that an earlier kernel left there turned dL/dSH of the dynamic
    model into NaN (seen with 7 bases, 5 views, T = 6; whether it shows depends on what ran before)."""
    test_sh_grad_views_elementwise_against_float64(deg, 5, 6, (1301, 1302), 7)


@pytest.mark.gpu
@pytest.mark.parametrize("deg,V,T,sizes,K", SGV_CASES[:6])
def test_sh_adam_views_elementwise_against_float64(deg, V, T, sizes, K):
    ns, nd = sizes
    sc, scene, vms, bts, dcol, scale, ref = _sgv_inputs(deg, V, T, ns, nd, K, seed=deg * 100 + V + T + K + 5)
    b1, b2, eps, step, lr_dc, lr_rest = 0.9, 0.999, 1e-15, 3, 2.5e-3, 1.25e-4
    gen = torch.Generator().manual_seed(deg + V)
    f64 = torch.float64
    bc1, bc2 = 1.0 - b1 ** step, 1.0 - b2 ** step
    st_args = []
    checks = []
    for tag, lo, m, sa in (("static", 0, ns, scene.st), ("dynamic", ns, nd, scene.dy)):
        a = _lib.RdgShAdam()
        if m:
            p0 = {"dc": sa.sh_dc.reshape(m, 3).clone(), "rest": sa.sh_rest.reshape(m, 45).clone()}
            g = {"dc": ref[lo:lo + m, 0], "rest": ref[lo:lo + m, 1:].reshape(m, 45)}
            mom = {}
            for part, w in (("dc", 3), ("rest", 45)):
                gm = g[part].abs().mean().item() + 1e-12
                m1 = (0.3 * gm * torch.randn(m, w, generator=gen)).float()
                m2 = ((gm * (0.5 + torch.rand(m, w, generator=gen))) ** 2).float()
                mom[part] = (m1.cuda(), m2.cuda())
                mn = b1 * m1.to(f64) + (1 - b1) * g[part]
                vn = b2 * m2.to(f64) + (1 - b2) * g[part] ** 2
                lr = lr_dc if part == "dc" else lr_rest
                dp = -lr / bc1 * mn / (vn.sqrt() / math.sqrt(bc2) + eps)
                checks.append((f"{tag}.{part}", p0[part], sa.sh_dc if part == "dc" else sa.sh_rest, mom[part], dp, mn, vn))
            a.exp_avg_dc, a.exp_avg_sq_dc = ptr(mom["dc"][0]), ptr(mom["dc"][1])
            a.exp_avg_rest, a.exp_avg_sq_rest = ptr(mom["rest"][0]), ptr(mom["rest"][1])
            a.lr_dc, a.lr_rest, a.step = lr_dc, lr_rest, step
        st_args.append(a)
    check(_lib.load().rdg_sh_adam_views(C.byref(engine._scene_struct(scene)), deg, V, ptr(vms), ptr(bts), ptr(dcol), scale,
                                        C.byref(st_args[0]), C.byref(st_args[1]), b1, b2, eps, _lib.stream_ptr()))
    row = []
    for name, p0, p_now, (m1, m2), dp, mn, vn in checks:
        # the parameter is stored in float32, whose rounding alone moves a 1e-6 step of a unit parameter by ~5 %: the float32
        # oracle (float64 step added in float32) carries the same rounding and is the yardstick where it misses the bar
        p0 = p0.cpu()
        p_now = p_now.reshape(p0.shape).cpu().to(f64)
        step32 = (p0 + dp.float()).to(f64) - p0.to(f64)
        _check(f"{name}.step", p_now - p0.to(f64), dp, step32, table=row)
        _check(f"{name}.m", m1.cpu(), mn, table=row)
        _check(f"{name}.v", m2.cpu(), vn, table=row)
    print(f"sh_adam_views deg {deg} V {V} T {T} {ns}+{nd} K {K}: " + "; ".join(row))


# --------------------------------------------------------------------------------- part 4: the bar has teeth (CPU) --

def test_elementwise_bar_rejects_what_the_normwise_bar_lets_through():
    """Three plausible kernel bugs applied to the float64 acc of a small ragged scene: the element-wise bar rejects each of
    them, while the norm-wise max|a-b| / max|b| <= 1e-3 that holds the per-Gaussian tensors end to end accepts some."""
    H, W = 45, 70                                               # 45 % 16 = 13: region 1 of the bottom tiles has 5 rows
    sc, cam = helpers.small_scene(1500, H, W, 6, seed=12, radius_px=2.5)
    acts = [a.detach().double() for a in helpers.activated_concat(sc, cam)]
    st = so.Settings(H, W, cam.tanfovx, cam.tanfovy, torch.tensor([0.1, 0.2, 0.3], dtype=torch.float64), 1.0,
                     cam.projection_matrix.t().contiguous().double(), 3)
    pp = so.preprocess(acts[0], acts[2], acts[3], acts[1], acts[4], None, cam.world_view_transform.t().contiguous().double(), st)
    bn = so.bin_tiles(pp, H, W)
    rec = {"xy": pp.xy.detach(), "conic": pp.conic.detach(), "opacity": pp.opacity.detach(), "rgb": pp.rgb.detach(),
           "depth": pp.depth.detach()}
    g = torch.Generator().manual_seed(1)
    up = (torch.randn(3, H, W, generator=g), 0.3 * torch.randn(1, H, W, generator=g), 0.2 * torch.randn(1, H, W, generator=g))
    acc, _ = _oracle_acc(rec, bn.local, bn.ranges, st.bg, H, W, up)
    # (a) region 1 of the bottom tiles dropped
    cut = 16 * (H // 16) + 8
    up_a = tuple(u.clone() for u in up)
    for u in up_a:
        u[:, cut:] = 0.0
    mut_a, _ = _oracle_acc(rec, bn.local, bn.ranges, st.bg, H, W, up_a)
    # (b) dB of the Gaussians with a radius of at most 3 px off by 1 %
    mut_b = acc.clone()
    small = pp.radii[pp.idx] <= 3
    assert int((small & pp.visible).sum()) > 10
    mut_b[small, 3] *= 1.01
    # (c) the 1 % of rows with the smallest non-zero |dL/dopacity| zeroed
    mut_c = acc.clone()
    nz = (acc[:, 5] != 0).nonzero().squeeze(1)
    k = max(1, nz.numel() // 100)
    mut_c[nz[acc[nz, 5].abs().argsort()[:k]], 5] = 0.0
    accepted = []
    for name, mut in (("region 1 of the bottom tiles dropped", mut_a), ("dB of small splats x 1.01", mut_b),
                      ("smallest 1 % of dL/dopacity zeroed", mut_c)):
        assert not bool(torch.equal(mut, acc)), name
        elem_ok = all(helpers.elementwise_ok(mut[:, c], acc[:, c])[0] for c in range(10))
        norm_ok = all(helpers.rel_err(mut[:, c], acc[:, c]) <= 1e-3 for c in range(10))
        assert not elem_ok, f"the element-wise bar accepts the mutant '{name}'"
        if norm_ok:
            accepted.append(name)
    assert accepted, "the norm-wise bar rejects all three mutants"
    print("accepted by the norm-wise bar only:", accepted)
