"""Host-side driver of one render (forward) and its backward through the C ABI.

Both public entry points sit on top of this module:
  * rodygs_b200.rasterizer  - the drop-in `GaussianRasterizer` boundary
    (/root/reference/src/trainer/renderer.py:50-101), activated + concatenated inputs;
  * rodygs_b200.dynamic     - the fused path on raw parameters of the static and the
    dynamic model (replaces rodygs.py:68-113 + rodygs_static.py:82-105 +
    rodygs_dynamic.py:122-138 + the render call).

PyTorch is plumbing here: it owns the device memory and the stream.  All compute
is in librodygs_b200.so; nothing in this file computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import Dict, Optional

import torch

from . import _lib
from ._lib import RdgBins, RdgGeom, RdgImage, RdgScene, RdgSceneGrad, RdgSet, RdgSetGrad, RdgView, check, ptr

TILE = 16
NACC = 12


class Config:
    """Process-wide knobs.

    sync_free: False (default) keeps the reference's behaviour of one host read of the
      duplicate count per forward (upstream reads `num_rendered` to size its binning
      buffers) and transparently re-bins with a larger buffer on overflow.  True never
      synchronises: the count stays on the device, buffers are sized from the high-water
      mark times `headroom`, and an overflow is raised at the next call.
    """
    sync_free: bool = False
    headroom: float = 1.25
    min_capacity: int = 1 << 16
    debug_keep_unsorted: bool = False   # tests: keep duplicateWithKeys' output
    debug_activated: bool = False       # tests: dump the activated parameters the kernel used
    # "tiles": tile-bucketed binning (per-tile shared-memory sort, rdg_bin_tiles) - the fast path.
    # "lsd":   scan + duplicateWithKeys + global LSD radix sort (rdg_bin); also produces the
    #          emission-order arrays (point_offsets, unsorted keys/values) that the tests pin.
    binning: str = "tiles"
    emit_sorted_keys: bool = True       # write the sorted 64-bit keys (only verification reads them)
    # Run-to-run reproducible backward pass (test mode, several times slower): the blend backward sums its per-region
    # partials as scaled 64-bit integers (rdg_blend_bwd_deterministic) and the per-Gaussian backward runs on one CTA so that
    # the cross-CTA atomics of dL/dV, dL/dtable, dL/dB(t) keep one order.  Also switched on by RDG_DETERMINISTIC=1.
    deterministic: bool = os.environ.get("RDG_DETERMINISTIC", "0") == "1"
    # set by SplatTrainStep.capture_forward_backward while a CUDA graph of the step is being captured (sync_free only): the
    # host-side look at the previous frame's duplicate count moves to CapturedStep.replay()
    capturing: bool = False
    capture_host = None                 # pinned [2] int32 that receives the captured step's duplicate count


config = Config()

# per-device duplicate-capacity state: {"cap": int, "pending": (pinned tensor, event) | None}
_capacity: Dict[int, dict] = {}


def _cap_state(device: torch.device, n: int) -> dict:
    st = _capacity.get(device.index)
    if st is None:
        st = {"cap": max(config.min_capacity, 4 * n), "pending": None}
        _capacity[device.index] = st
    return st


def reset_capacity():
    _capacity.clear()


def _check_pending(st: dict):
    """Look at the duplicate count of an earlier sync-free call (already finished)."""
    pend = st["pending"]
    if pend is None:
        return
    host, ev, cap_used = pend
    if ev is not None:
        ev.synchronize()
    st["pending"] = None
    d = int(host[0])
    if d > cap_used:
        st["cap"] = int(d * config.headroom) + 1
        raise RuntimeError(
            f"rodygs_b200: a previous sync-free render produced {d} tile instances but its buffers held "
            f"{cap_used}; that frame was truncated. Capacity is now {st['cap']}; re-run the step "
            "(or set rodygs_b200.config.sync_free = False).")
    if d * config.headroom > st["cap"]:
        st["cap"] = int(d * config.headroom) + 1


@dataclass
class SetArgs:
    xyz: torch.Tensor
    scaling: torch.Tensor
    rotation: torch.Tensor
    opacity: torch.Tensor
    sh_dc: Optional[torch.Tensor]
    sh_rest: Optional[torch.Tensor]
    sh_dc_stride: int = 3
    sh_rest_stride: int = 45
    sh_rest_offset: int = 0     # float offset of sh_rest inside its tensor (3 for a cat'ed [n,16,3])

    def n(self) -> int:
        return 0 if self.xyz is None else self.xyz.shape[0]


@dataclass
class SceneArgs:
    st: Optional[SetArgs]
    dy: Optional[SetArgs] = None
    raw: bool = False
    colors_precomp: Optional[torch.Tensor] = None
    use_deform: bool = False
    motion_coeff: Optional[torch.Tensor] = None   # [nd, K]
    time_ind: Optional[torch.Tensor] = None       # [nd] int32
    basis_t: Optional[torch.Tensor] = None        # [K,7]
    table: Optional[torch.Tensor] = None          # [T,K,7]
    spatial_lr_scale: float = 1.0
    frame_order: Optional[torch.Tensor] = None    # [nd] int32, stable argsort(time_ind)
    frame_offsets: Optional[torch.Tensor] = None  # [T+1] int32

    def counts(self):
        ns = self.st.n() if self.st is not None else 0
        nd = self.dy.n() if self.dy is not None else 0
        return ns, nd


@dataclass
class ViewArgs:
    height: int
    width: int
    tanfovx: float
    tanfovy: float
    scale_modifier: float
    sh_degree: int
    viewmatrix: torch.Tensor   # [4,4] glm storage, contiguous
    projmatrix: torch.Tensor
    bg: torch.Tensor
    enable_cov_grad: bool = True
    enable_sh_grad: bool = True


@dataclass
class FwdState:
    """Everything the backward pass needs (kept alive by the autograd ctx)."""
    scene: SceneArgs
    view: ViewArgs
    n: int
    geom: dict
    vals_sorted: torch.Tensor
    ranges: torch.Tensor
    num_rendered: torch.Tensor
    final_T: torch.Tensor
    n_contrib: torch.Tensor
    d_cap: int
    extras: dict = field(default_factory=dict)


def _set_struct(s: Optional[SetArgs]) -> RdgSet:
    out = RdgSet()
    if s is None or s.n() == 0:
        return out
    out.xyz = ptr(s.xyz)
    out.scaling = ptr(s.scaling)
    out.rotation = ptr(s.rotation)
    out.opacity = ptr(s.opacity)
    out.sh_dc = ptr(s.sh_dc)
    out.sh_rest = None if s.sh_rest is None else s.sh_rest.data_ptr() + 4 * s.sh_rest_offset
    out.sh_dc_stride = s.sh_dc_stride
    out.sh_rest_stride = s.sh_rest_stride
    return out


def _scene_struct(sc: SceneArgs) -> RdgScene:
    ns, nd = sc.counts()
    out = RdgScene()
    out.n_static, out.n_dynamic = ns, nd
    out.st = _set_struct(sc.st)
    out.dy = _set_struct(sc.dy)
    out.raw = 1 if sc.raw else 0
    out.colors_precomp = ptr(sc.colors_precomp)
    out.use_deform = 1 if (sc.use_deform and nd > 0) else 0
    if out.use_deform:
        out.num_basis = sc.motion_coeff.shape[-1]
        out.num_times = sc.table.shape[0]
        out.motion_coeff = ptr(sc.motion_coeff)
        out.time_ind = ptr(sc.time_ind)
        out.basis_t = ptr(sc.basis_t)
        out.table = ptr(sc.table)
        out.frame_order = ptr(sc.frame_order)
        out.frame_offsets = ptr(sc.frame_offsets)
    out.spatial_lr_scale = float(sc.spatial_lr_scale)
    return out


def _view_struct(v: ViewArgs) -> RdgView:
    out = RdgView()
    out.height, out.width = int(v.height), int(v.width)
    out.tanfovx, out.tanfovy = float(v.tanfovx), float(v.tanfovy)
    out.scale_modifier = float(v.scale_modifier)
    out.sh_degree = int(v.sh_degree)
    out.enable_cov_grad = 1 if v.enable_cov_grad else 0
    out.enable_sh_grad = 1 if v.enable_sh_grad else 0
    out.viewmatrix = ptr(v.viewmatrix)
    out.projmatrix = ptr(v.projmatrix)
    out.bg = ptr(v.bg)
    return out


def _geom_struct(g: dict) -> RdgGeom:
    out = RdgGeom()
    out.radii = ptr(g["radii"])
    out.tiles_touched = ptr(g["tiles_touched"])
    out.p0, out.p1, out.p2 = ptr(g["p0"]), ptr(g["p1"]), ptr(g["p2"])
    out.clamped = ptr(g["clamped"])
    out.dbg_activated = ptr(g.get("dbg_activated"))
    out.tile_count = ptr(g.get("tile_count"))
    return out


_csr_cache: Dict[tuple, tuple] = {}


def frame_csr(time_ind: torch.Tensor, num_times: int):
    """CSR of the dynamic Gaussians by birth frame: (order [nd] int32, offsets [T+1] int32).
    Built on the device once per `time_ind` tensor (it only changes on densification) and cached.  The cache entry keeps
    the tensor itself alive and is only reused for that very object at the same version: a recycled address (temporaries
    of the caching allocator) or an in-place rewrite through a raw pointer cannot alias a stale entry - callers that
    write time_ind through the C ABI (densification) build a new tensor, SplatTrainStep keeps its own CSR."""
    key = (id(time_ind), int(num_times))
    hit = _csr_cache.get(key)
    if hit is not None and hit[0] is time_ind and hit[1] == time_ind._version:
        return hit[2]
    if len(_csr_cache) > 16:
        _csr_cache.clear()
    ti = time_ind.long()
    sorted_ti, order = torch.sort(ti, stable=True)
    offsets = torch.searchsorted(sorted_ti, torch.arange(num_times + 1, device=ti.device))
    out = (order.to(torch.int32).contiguous(), offsets.to(torch.int32).contiguous())
    _csr_cache[key] = (time_ind, time_ind._version, out)
    return out


def frame_csr_of(time_ind: torch.Tensor, num_times: int):
    """(time_ind as contiguous int32, order, offsets) for a `gaussian_to_time_ind` of any integer dtype (the reference keeps
    it as int64, rodygs_dynamic.py:58-77), cached on the caller's tensor object like frame_csr."""
    key = (id(time_ind), int(num_times), "any")
    hit = _csr_cache.get(key)
    if hit is not None and hit[0] is time_ind and hit[1] == time_ind._version:
        return hit[2]
    ti32 = time_ind if (time_ind.dtype == torch.int32 and time_ind.is_contiguous()) else time_ind.to(torch.int32).contiguous()
    order, offsets = frame_csr(ti32, num_times)
    out = (ti32, order, offsets)
    _csr_cache[key] = (time_ind, time_ind._version, out)
    return out


def tiles_of(h: int, w: int) -> int:
    return ((h + TILE - 1) // TILE) * ((w + TILE - 1) // TILE)


def render_forward(scene: SceneArgs, view: ViewArgs, keep_for_backward: bool = True, stage_hook=None):
    """preprocess -> bin -> blend.  Returns (color, depth, alpha, radii, FwdState)."""
    lib = _lib.load()
    ns, nd = scene.counts()
    n = ns + nd
    dev = view.viewmatrix.device
    if dev.type != "cuda":
        raise RuntimeError("rodygs_b200 runs on CUDA tensors only (no CPU fallback)")
    stream = _lib.stream_ptr()
    H, W = int(view.height), int(view.width)
    f32 = dict(dtype=torch.float32, device=dev)
    geom = {
        "radii": torch.empty(n, dtype=torch.int32, device=dev),
        "tiles_touched": torch.empty(n, dtype=torch.int32, device=dev),
        "p0": torch.empty(n, 4, **f32), "p1": torch.empty(n, 4, **f32), "p2": torch.empty(n, 2, **f32),
        "clamped": torch.empty(n, dtype=torch.uint8, device=dev),
    }
    if config.debug_activated:
        geom["dbg_activated"] = torch.zeros(n, 11, **f32)
    use_tiles = config.binning == "tiles" and not config.debug_keep_unsorted
    if use_tiles:
        geom["tile_count"] = torch.empty(tiles_of(H, W) + 1, dtype=torch.int32, device=dev)
    sc_s, vw_s, gm_s = _scene_struct(scene), _view_struct(view), _geom_struct(geom)
    check(lib.rdg_preprocess_fwd(C.byref(sc_s), C.byref(vw_s), C.byref(gm_s), stream))
    if stage_hook:
        stage_hook("preprocess_fwd")

    st = _cap_state(dev, n)
    if not config.capturing:
        _check_pending(st)
    ntiles = tiles_of(H, W)
    ranges = torch.empty(ntiles, 2, dtype=torch.int32, device=dev)
    point_offsets = torch.empty(n, dtype=torch.int32, device=dev)
    num_rendered = torch.empty(2, dtype=torch.int32, device=dev)
    extras = {}
    while True:
        d_cap = int(st["cap"])
        want_keys = config.emit_sorted_keys or not use_tiles
        keys = torch.empty(d_cap, dtype=torch.int64, device=dev) if want_keys else None
        vals = torch.empty(d_cap, dtype=torch.int32, device=dev)
        # region lists of the blend kernels (two 16x8 regions per tile; rdg_blend_fwd writes, rdg_blend_bwd reads)
        region_ids = torch.empty(2 * d_cap, dtype=torch.int32, device=dev)
        region_masks = torch.empty(2 * d_cap, dtype=torch.uint8, device=dev)
        region_count = torch.empty(2 * ntiles, dtype=torch.int32, device=dev)
        ws_bytes = int((lib.rdg_bin_tiles_workspace_bytes if use_tiles else lib.rdg_bin_workspace_bytes)(n, d_cap, H, W))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        bins = RdgBins()
        bins.keys_sorted, bins.vals_sorted = ptr(keys), ptr(vals)
        bins.ranges, bins.point_offsets, bins.num_rendered = ptr(ranges), ptr(point_offsets), ptr(num_rendered)
        bins.region_ids, bins.region_masks, bins.region_count = ptr(region_ids), ptr(region_masks), ptr(region_count)
        bins.region_stride = d_cap
        if config.debug_keep_unsorted:
            extras["keys_unsorted"] = torch.empty(d_cap, dtype=torch.int64, device=dev)
            extras["vals_unsorted"] = torch.empty(d_cap, dtype=torch.int32, device=dev)
            bins.keys_unsorted, bins.vals_unsorted = ptr(extras["keys_unsorted"]), ptr(extras["vals_unsorted"])
        check((lib.rdg_bin_tiles if use_tiles else lib.rdg_bin)(n, C.byref(gm_s), H, W, d_cap, C.byref(bins), ptr(ws),
                                                                ws_bytes, stream))
        if config.sync_free:
            # (under graph capture the pinned buffer was allocated beforehand: no cudaHostAlloc inside a capture)
            host = config.capture_host if config.capturing else torch.empty(2, dtype=torch.int32, pin_memory=True)
            host.copy_(num_rendered, non_blocking=True)
            ev = None
            if not config.capturing:
                ev = torch.cuda.Event()
                ev.record()
            st["pending"] = (host, ev, d_cap)
            break
        d = int(num_rendered[0].item())          # the reference's one host read per forward
        if d <= d_cap:
            if d * config.headroom > d_cap:
                st["cap"] = int(d * config.headroom) + 1
            break
        st["cap"] = int(d * config.headroom) + 1  # overflow: re-bin with a larger buffer

    if stage_hook:
        stage_hook("bin")
    color = torch.empty(3, H, W, **f32)
    depth = torch.empty(1, H, W, **f32)
    alpha = torch.empty(1, H, W, **f32)
    final_T = torch.empty(H, W, **f32)
    n_contrib = torch.empty(H, W, dtype=torch.int32, device=dev)
    img = RdgImage()
    img.color, img.depth, img.alpha, img.final_T, img.n_contrib = ptr(color), ptr(depth), ptr(alpha), ptr(final_T), ptr(n_contrib)
    check(lib.rdg_blend_fwd(n, C.byref(gm_s), C.byref(bins), C.byref(vw_s), C.byref(img), stream))
    if stage_hook:
        stage_hook("blend_fwd")

    extras.update({"keys_sorted": keys, "point_offsets": point_offsets, "region_ids": region_ids, "region_masks": region_masks,
                   "region_count": region_count})
    state = FwdState(scene=scene, view=view, n=n, geom=geom, vals_sorted=vals, ranges=ranges,
                     num_rendered=num_rendered, final_T=final_T, n_contrib=n_contrib, d_cap=d_cap, extras=extras)
    return color, depth, alpha, geom["radii"], state


VIEWS_PER_LAUNCH = 8   # rdg_preprocess_fwd_views


def render_views(scene: SceneArgs, views, basis_ts: Optional[torch.Tensor], stage_hook=None):
    """render_forward of every view in `views` (ViewArgs sharing height, width, sh_degree and scale_modifier; scene.basis_t
    None, B(t) of view v = basis_ts[v]), with the same bits.  Passes of up to 8 views: ONE rdg_preprocess_fwd_views, ONE host
    read of the pass's duplicate counts (sums of each view's tile counts), then binning buffers of exactly that size and
    rdg_bin_tiles + rdg_blend_fwd per view, so nothing overflows or is re-binned.  The duplicate-capacity state
    (_capacity, a pending sync-free count) is neither read nor changed.
    Returns (color [V,3,H,W], depth [V,1,H,W], alpha [V,1,H,W], radii [V,N] int32)."""
    lib = _lib.load()
    ns, nd = scene.counts()
    n = ns + nd
    V = len(views)
    dev = views[0].viewmatrix.device
    if dev.type != "cuda":
        raise RuntimeError("rodygs_b200 runs on CUDA tensors only (no CPU fallback)")
    stream = _lib.stream_ptr()
    H, W = int(views[0].height), int(views[0].width)
    ntiles = tiles_of(H, W)
    f32 = dict(dtype=torch.float32, device=dev)
    color = torch.empty(V, 3, H, W, **f32)
    depth = torch.empty(V, 1, H, W, **f32)
    alpha = torch.empty(V, 1, H, W, **f32)
    radii = torch.empty(V, n, dtype=torch.int32, device=dev)
    sc_s = _scene_struct(scene)
    final_T = torch.empty(H, W, **f32)
    n_contrib = torch.empty(H, W, dtype=torch.int32, device=dev)
    ranges = torch.empty(ntiles, 2, dtype=torch.int32, device=dev)
    num_rendered = torch.empty(2, dtype=torch.int32, device=dev)
    region_count = torch.empty(2 * ntiles, dtype=torch.int32, device=dev)
    for lo in range(0, V, VIEWS_PER_LAUNCH):
        pv = views[lo:lo + VIEWS_PER_LAUNCH]
        k = len(pv)
        # zeroed here as well: without Gaussians the kernel returns before it zeroes them, and the counts must still read 0
        tile_count = torch.zeros(k, ntiles + 1, dtype=torch.int32, device=dev)
        geoms = [{"radii": radii[lo + j], "tiles_touched": torch.empty(n, dtype=torch.int32, device=dev),
                  "p0": torch.empty(n, 4, **f32), "p1": torch.empty(n, 4, **f32), "p2": torch.empty(n, 2, **f32),
                  "clamped": torch.empty(n, dtype=torch.uint8, device=dev), "tile_count": tile_count[j]} for j in range(k)]
        vw_s = (RdgView * k)(*[_view_struct(v) for v in pv])
        gm_s = (RdgGeom * k)(*[_geom_struct(g) for g in geoms])
        bts = None if basis_ts is None else basis_ts[lo:lo + k].contiguous()
        check(lib.rdg_preprocess_fwd_views(C.byref(sc_s), ptr(bts), k, vw_s, gm_s, stream))
        if stage_hook:
            stage_hook("preprocess_fwd")
        counts = tile_count[:, :ntiles].sum(1).tolist()          # the pass's one host read
        for j in range(k):
            d_cap = max(int(counts[j]), 1)
            vals = torch.empty(d_cap, dtype=torch.int32, device=dev)
            region_ids = torch.empty(2 * d_cap, dtype=torch.int32, device=dev)
            region_masks = torch.empty(2 * d_cap, dtype=torch.uint8, device=dev)
            ws_bytes = int(lib.rdg_bin_tiles_workspace_bytes(n, d_cap, H, W))
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            bins = RdgBins()
            bins.vals_sorted, bins.ranges, bins.num_rendered = ptr(vals), ptr(ranges), ptr(num_rendered)
            bins.region_ids, bins.region_masks, bins.region_count = ptr(region_ids), ptr(region_masks), ptr(region_count)
            bins.region_stride = d_cap
            check(lib.rdg_bin_tiles(n, C.byref(gm_s[j]), H, W, d_cap, C.byref(bins), ptr(ws), ws_bytes, stream))
            img = RdgImage()
            v = lo + j
            img.color, img.depth, img.alpha = ptr(color[v]), ptr(depth[v]), ptr(alpha[v])
            img.final_T, img.n_contrib = ptr(final_T), ptr(n_contrib)
            check(lib.rdg_blend_fwd(n, C.byref(gm_s[j]), C.byref(bins), C.byref(vw_s[j]), C.byref(img), stream))
        if stage_hook:
            stage_hook("bin_blend")
    return color, depth, alpha, radii


TARGETS_PER_PASS = 8   # engine.track: bounds the blended maps at 8 x 3 x H x W floats


def track(scene: SceneArgs, view_src: ViewArgs, basis_t_src: Optional[torch.Tensor], target_viewmats: torch.Tensor,
          target_projmats: torch.Tensor, target_basis_ts: Optional[torch.Tensor], points: Optional[torch.Tensor] = None,
          stage_hook=None, keep_maps: bool = False):
    """Where each pixel (or query point) of the source render goes at M target camera-times (INTEGRATION.md §10).
    scene.basis_t None; B(t_s) = basis_t_src, B(t_m) = target_basis_ts[m] (both None without deformation);
    target_viewmats / target_projmats [M, 4, 4] glm storage; points None or [P, 2] pixel coordinates.

    One rdg_preprocess_fwd of the source view, ONE host read of its duplicate count, exactly sized binning buffers
    (rdg_bin_tiles); then targets in passes of at most 8: per target rdg_track_attrs + rdg_blend_fwd (zero background) into
    S [k, 3, H, W], and one rdg_track_project per pass.  The duplicate-capacity state (_capacity, a pending sync-free count)
    is neither read nor changed.  stage_hook(name) is called after "source" (preprocess + binning) and after every "attrs",
    "blend" and "project" launch.  keep_maps (tests): also return S_m of every target [M, 3, H, W] and mu_k(t_m)
    [M, N, 3] (rdg_track_attrs' positions_out).
    Returns dense (xy [M, 2, H, W], depth [M, 1, H, W], alpha [1, H, W]) or sparse (xy [M, P, 2], depth [M, P],
    alpha [P]), then (S, positions) with keep_maps."""
    lib = _lib.load()
    ns, nd = scene.counts()
    n = ns + nd
    M = target_viewmats.shape[0]
    dev = view_src.viewmatrix.device
    if dev.type != "cuda":
        raise RuntimeError("rodygs_b200 runs on CUDA tensors only (no CPU fallback)")
    stream = _lib.stream_ptr()
    H, W = int(view_src.height), int(view_src.width)
    ntiles = tiles_of(H, W)
    f32 = dict(dtype=torch.float32, device=dev)
    # the source render: its records, bins and alpha are shared by every target
    geom = {"radii": torch.empty(n, dtype=torch.int32, device=dev), "tiles_touched": torch.empty(n, dtype=torch.int32, device=dev),
            "p0": torch.empty(n, 4, **f32), "p1": torch.empty(n, 4, **f32), "p2": torch.empty(n, 2, **f32),
            "clamped": torch.empty(n, dtype=torch.uint8, device=dev),
            # zeroed here as well: without Gaussians preprocess returns before it zeroes them
            "tile_count": torch.zeros(ntiles + 1, dtype=torch.int32, device=dev)}
    sc_s, gm_s = _scene_struct(scene), _geom_struct(geom)
    sc_s.basis_t = ptr(basis_t_src) if sc_s.use_deform else None
    check(lib.rdg_preprocess_fwd(C.byref(sc_s), C.byref(_view_struct(view_src)), C.byref(gm_s), stream))
    sc_s.basis_t = None                                          # rdg_track_attrs takes B(t_m) on its own
    d_cap = max(int(geom["tile_count"][:ntiles].sum()), 1)      # the call's one host read
    vals = torch.empty(d_cap, dtype=torch.int32, device=dev)
    ranges = torch.empty(ntiles, 2, dtype=torch.int32, device=dev)
    num_rendered = torch.empty(2, dtype=torch.int32, device=dev)
    region_ids = torch.empty(2 * d_cap, dtype=torch.int32, device=dev)
    region_masks = torch.empty(2 * d_cap, dtype=torch.uint8, device=dev)
    region_count = torch.empty(2 * ntiles, dtype=torch.int32, device=dev)
    ws_bytes = int(lib.rdg_bin_tiles_workspace_bytes(n, d_cap, H, W))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    bins = RdgBins()
    bins.vals_sorted, bins.ranges, bins.num_rendered = ptr(vals), ptr(ranges), ptr(num_rendered)
    bins.region_ids, bins.region_masks, bins.region_count = ptr(region_ids), ptr(region_masks), ptr(region_count)
    bins.region_stride = d_cap
    check(lib.rdg_bin_tiles(n, C.byref(gm_s), H, W, d_cap, C.byref(bins), ptr(ws), ws_bytes, stream))
    if stage_hook:
        stage_hook("source")

    zero_bg = torch.zeros(3, **f32)
    vw_blend = _view_struct(view_src)
    vw_blend.bg = ptr(zero_bg)
    alpha = torch.empty(1, H, W, **f32)
    blend_depth = torch.empty(1, H, W, **f32)
    final_T = torch.empty(H, W, **f32)
    n_contrib = torch.empty(H, W, dtype=torch.int32, device=dev)
    vms, pms = target_viewmats.contiguous(), target_projmats.contiguous()
    sparse = points is not None
    P = points.shape[0] if sparse else 0
    if sparse:
        xy, depth = torch.empty(M, P, 2, **f32), torch.empty(M, P, **f32)
        alpha_pts = torch.empty(P, **f32)
    else:
        xy, depth = torch.empty(M, 2, H, W, **f32), torch.empty(M, 1, H, W, **f32)
    S_all = torch.empty(M, 3, H, W, **f32) if keep_maps else None
    positions = torch.empty(M, n, 3, **f32) if keep_maps else None
    S_pass = None if keep_maps else torch.empty(min(M, TARGETS_PER_PASS), 3, H, W, **f32)
    for lo in range(0, M, TARGETS_PER_PASS):
        k = min(TARGETS_PER_PASS, M - lo)
        S = S_all[lo:lo + k] if keep_maps else S_pass[:k]
        for j in range(k):
            m = lo + j
            bt = None if target_basis_ts is None or not sc_s.use_deform else target_basis_ts[m]
            check(lib.rdg_track_attrs(C.byref(sc_s), ptr(bt), C.byref(gm_s), ptr(positions[m]) if keep_maps else None, stream))
            if stage_hook:
                stage_hook("attrs")
            img = RdgImage()
            img.color, img.depth, img.alpha = ptr(S[j]), ptr(blend_depth), ptr(alpha)
            img.final_T, img.n_contrib = ptr(final_T), ptr(n_contrib)
            check(lib.rdg_blend_fwd(n, C.byref(gm_s), C.byref(bins), C.byref(vw_blend), C.byref(img), stream))
            if stage_hook:
                stage_hook("blend")
        if not sparse:
            check(lib.rdg_track_project(ptr(S), ptr(alpha), k, H, W, ptr(vms[lo:lo + k]), ptr(pms[lo:lo + k]), None, 0,
                                        ptr(xy[lo:lo + k]), ptr(depth[lo:lo + k]), None, stream))
        elif P > 0:                                              # without query points the empty outputs have no storage
            check(lib.rdg_track_project(ptr(S), ptr(alpha), k, H, W, ptr(vms[lo:lo + k]), ptr(pms[lo:lo + k]), ptr(points), P,
                                        ptr(xy[lo:lo + k]), ptr(depth[lo:lo + k]), ptr(alpha_pts), stream))
        if stage_hook:
            stage_hook("project")
    out = (xy, depth, alpha_pts if sparse else alpha)
    return out + (S_all, positions) if keep_maps else out


@dataclass
class SetGrads:
    xyz: Optional[torch.Tensor] = None
    scaling: Optional[torch.Tensor] = None
    rotation: Optional[torch.Tensor] = None
    opacity: Optional[torch.Tensor] = None
    sh_dc: Optional[torch.Tensor] = None
    sh_rest: Optional[torch.Tensor] = None
    sh_rest_offset: int = 0


@dataclass
class SceneGrads:
    st: SetGrads = field(default_factory=SetGrads)
    dy: SetGrads = field(default_factory=SetGrads)
    colors_precomp: Optional[torch.Tensor] = None
    means2D: Optional[torch.Tensor] = None
    viewmatrix: Optional[torch.Tensor] = None   # must be zero-initialised
    motion_coeff: Optional[torch.Tensor] = None
    table: Optional[torch.Tensor] = None        # must be zero-initialised
    basis_t: Optional[torch.Tensor] = None      # must be zero-initialised
    g7_scratch: Optional[torch.Tensor] = None   # [nd,8] scratch (allocated on demand)
    dcolor: Optional[torch.Tensor] = None       # [N,3] factors of dL/dSH for the data-parallel exchange
    sm_queue: Optional[torch.Tensor] = None     # [4] int32 scratch: SM-partitioned per-Gaussian backward (data parallel)
    dcolor_mc: int = 0                          # multicast address of this view's block of the gathered factors (0: none)
    dcolor_stream: Optional[torch.cuda.Stream] = None   # side stream for the multicast kernel (its stores take NVLink time)


def _setgrad_struct(g: SetGrads) -> RdgSetGrad:
    out = RdgSetGrad()
    out.xyz, out.scaling, out.rotation, out.opacity = ptr(g.xyz), ptr(g.scaling), ptr(g.rotation), ptr(g.opacity)
    out.sh_dc = ptr(g.sh_dc)
    out.sh_rest = None if g.sh_rest is None else g.sh_rest.data_ptr() + 4 * g.sh_rest_offset
    return out


def render_backward(state: FwdState, dL_dcolor, dL_ddepth, dL_dalpha, grads: SceneGrads, stage_hook=None,
                    after_blend=None, after_model=None, bwd_plan=None):
    """blend backward -> preprocess backward.  Writes into the tensors of `grads`.
    after_blend: data-parallel mode - called as soon as grads.dcolor (the factors of dL/dSH) is final, i.e.
    right after the blend backward, so that their all-gather overlaps the per-Gaussian backward.
    after_model: data-parallel mode - the per-Gaussian backward runs as one launch per model (dynamic first: it is the
    larger gradient range) and after_model("dynamic") / after_model("static") is called right after each, so that the
    all-reduce of one model's range runs under the other model's kernel.
    bwd_plan: a finer schedule for the same - a sequence of (models, part, parts, dtable_mode, piece) launches
    (RdgSceneGrad.models / part / parts / dtable_mode); after_model(piece) is called after each."""
    lib = _lib.load()
    dev = state.view.viewmatrix.device
    stream = _lib.stream_ptr()
    n = state.n
    acc = torch.zeros(max(n, 1), NACC, dtype=torch.float32, device=dev)
    sc_s, vw_s, gm_s = _scene_struct(state.scene), _view_struct(state.view), _geom_struct(state.geom)
    bins = RdgBins()
    bins.vals_sorted, bins.ranges, bins.num_rendered = ptr(state.vals_sorted), ptr(state.ranges), ptr(state.num_rendered)
    bins.region_ids, bins.region_masks = ptr(state.extras["region_ids"]), ptr(state.extras["region_masks"])
    bins.region_count, bins.region_stride = ptr(state.extras["region_count"]), state.d_cap
    img = RdgImage()
    img.final_T, img.n_contrib = ptr(state.final_T), ptr(state.n_contrib)

    def c(t):
        return None if t is None else t.contiguous()

    dL_dcolor, dL_ddepth, dL_dalpha = c(dL_dcolor), c(dL_ddepth), c(dL_dalpha)
    _lib.set_tunable("deterministic", 1 if config.deterministic else 0)
    if config.deterministic:
        nb = int(lib.rdg_blend_bwd_deterministic_scratch_bytes(n))
        scratch = torch.empty(max(nb, 8), dtype=torch.uint8, device=dev)
        check(lib.rdg_blend_bwd_deterministic(n, C.byref(gm_s), C.byref(bins), C.byref(vw_s), C.byref(img), ptr(dL_dcolor),
                                              ptr(dL_ddepth), ptr(dL_dalpha), ptr(acc), ptr(scratch), nb, stream))
    else:
        check(lib.rdg_blend_bwd(n, C.byref(gm_s), C.byref(bins), C.byref(vw_s), C.byref(img),
                                ptr(dL_dcolor), ptr(dL_ddepth), ptr(dL_dalpha), ptr(acc), stream))
    early = after_blend is not None and grads.dcolor is not None and state.scene.colors_precomp is None
    if early:
        if grads.dcolor_mc:
            # NVLS: the factors go straight into every rank's gathered buffer (multicast stores).  The kernel lasts as long as
            # the NVLink transfer (its stores must be acknowledged), so it runs on a side stream beside the per-Gaussian backward
            side = grads.dcolor_stream
            if side is not None:
                ev = torch.cuda.Event()
                ev.record()
                side.wait_event(ev)
                acc.record_stream(side)
                state.geom["clamped"].record_stream(side)
                check(lib.rdg_dcolor_multicast(n, ptr(acc), ptr(state.geom["clamped"]), grads.dcolor_mc, side.cuda_stream))
            else:
                check(lib.rdg_dcolor_multicast(n, ptr(acc), ptr(state.geom["clamped"]), grads.dcolor_mc, stream))
        else:
            check(lib.rdg_dcolor_from_acc(n, ptr(acc), ptr(state.geom["clamped"]), ptr(grads.dcolor), stream))
        after_blend()
    if stage_hook:
        stage_hook("blend_bwd")
    g = RdgSceneGrad()
    g.st, g.dy = _setgrad_struct(grads.st), _setgrad_struct(grads.dy)
    g.colors_precomp, g.means2D, g.viewmatrix = ptr(grads.colors_precomp), ptr(grads.means2D), ptr(grads.viewmatrix)
    g.motion_coeff, g.table, g.basis_t = ptr(grads.motion_coeff), ptr(grads.table), ptr(grads.basis_t)
    g.dcolor = None if early else ptr(grads.dcolor)
    g.sm_queue = ptr(grads.sm_queue)
    if state.scene.use_deform and state.scene.frame_order is not None and grads.table is not None:
        if grads.g7_scratch is None:
            grads.g7_scratch = torch.empty(state.scene.motion_coeff.shape[0], 8, dtype=torch.float32, device=dev)
        g.g7_scratch = ptr(grads.g7_scratch)
    ns, nd = state.scene.counts()
    if after_model is not None and ns > 0 and nd > 0:
        # (models, part, parts, dtable_mode, piece name): one launch per piece, after_model(piece) after each
        plan = bwd_plan or ((2, 0, 1, 0, "dynamic"), (1, 0, 1, 0, "static"))
        for models, part, parts, dtable_mode, piece in plan:
            g.models, g.part, g.parts, g.dtable_mode = models, part, parts, dtable_mode
            check(lib.rdg_preprocess_bwd(C.byref(sc_s), C.byref(vw_s), C.byref(gm_s), ptr(acc), C.byref(g), stream))
            after_model(piece)
    else:
        g.models = 0
        check(lib.rdg_preprocess_bwd(C.byref(sc_s), C.byref(vw_s), C.byref(gm_s), ptr(acc), C.byref(g), stream))
        if after_model is not None:
            for piece in ("dynamic", "static") if nd > 0 else ("static", "dynamic"):
                after_model(piece)
    if stage_hook:
        stage_hook("preprocess_bwd")
    return acc
