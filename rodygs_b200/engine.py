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
from typing import Dict, List, Optional

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
    bins: Optional[RdgBins] = None    # the RdgBins the forward filled (its buffers are the tensors above)


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


def _image_struct(color, depth, alpha, final_T, n_contrib) -> RdgImage:
    out = RdgImage()
    out.color, out.depth, out.alpha, out.final_T, out.n_contrib = ptr(color), ptr(depth), ptr(alpha), ptr(final_T), ptr(n_contrib)
    return out


def _alloc_geom(n: int, dev: torch.device, radii: Optional[torch.Tensor] = None,
                tile_count: Optional[torch.Tensor] = None) -> dict:
    """The per-Gaussian records rdg_preprocess_fwd writes for one view, as the dict _geom_struct reads.  radii [n] int32 and
    tile_count [tiles + 1] int32 may be the caller's (render_views hands in rows of its [V, n] / [k, tiles + 1] outputs);
    without a tile_count the records have none (rdg_bin needs none)."""
    f32 = dict(dtype=torch.float32, device=dev)
    geom = {"radii": torch.empty(n, dtype=torch.int32, device=dev) if radii is None else radii,
            "tiles_touched": torch.empty(n, dtype=torch.int32, device=dev),
            "p0": torch.empty(n, 4, **f32), "p1": torch.empty(n, 4, **f32), "p2": torch.empty(n, 2, **f32),
            "clamped": torch.empty(n, dtype=torch.uint8, device=dev)}
    if tile_count is not None:
        geom["tile_count"] = tile_count
    return geom


class Bins:
    """The buffers of one frame's binning at duplicate capacity `cap` and the RdgBins over them (`s`).

    ranges [tiles, 2], num_rendered [2] and region_count [2 * tiles] are frame-sized and the caller's: render_views and the
    pose loop keep them across views and re-allocations.  Allocated here at `cap`: vals, keys (keys=True), the region lists
    of the blend kernels (two 16x8 regions per tile, region_stride = cap; rdg_blend_fwd writes them, rdg_blend_bwd reads
    them) and the binning workspace.  bin() runs rdg_bin_tiles or, with lsd, rdg_bin (scan + duplicateWithKeys + global LSD
    radix sort), which also needs the keys and point_offsets [n], and under config.debug_keep_unsorted keeps
    duplicateWithKeys' output in keys_unsorted / vals_unsorted."""

    def __init__(self, n: int, H: int, W: int, cap: int, ranges: torch.Tensor, num_rendered: torch.Tensor,
                 region_count: torch.Tensor, keys: bool = False, lsd: bool = False,
                 point_offsets: Optional[torch.Tensor] = None):
        lib = _lib.load()
        dev = ranges.device
        self.n, self.H, self.W, self.cap, self.lsd = n, H, W, cap, lsd
        self.keys = torch.empty(cap, dtype=torch.int64, device=dev) if keys or lsd else None
        self.vals = torch.empty(cap, dtype=torch.int32, device=dev)
        self.region_ids = torch.empty(2 * cap, dtype=torch.int32, device=dev)
        self.region_masks = torch.empty(2 * cap, dtype=torch.uint8, device=dev)
        self.ws_bytes = int((lib.rdg_bin_workspace_bytes if lsd else lib.rdg_bin_tiles_workspace_bytes)(n, cap, H, W))
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        s = RdgBins()
        s.keys_sorted, s.vals_sorted = ptr(self.keys), ptr(self.vals)
        s.ranges, s.point_offsets, s.num_rendered = ptr(ranges), ptr(point_offsets), ptr(num_rendered)
        s.region_ids, s.region_masks, s.region_count = ptr(self.region_ids), ptr(self.region_masks), ptr(region_count)
        s.region_stride = cap
        self.keys_unsorted = self.vals_unsorted = None
        if lsd and config.debug_keep_unsorted:
            self.keys_unsorted = torch.empty(cap, dtype=torch.int64, device=dev)
            self.vals_unsorted = torch.empty(cap, dtype=torch.int32, device=dev)
            s.keys_unsorted, s.vals_unsorted = ptr(self.keys_unsorted), ptr(self.vals_unsorted)
        self.s = s

    def bin(self, gm_s: RdgGeom):
        lib = _lib.load()
        check((lib.rdg_bin if self.lsd else lib.rdg_bin_tiles)(self.n, C.byref(gm_s), self.H, self.W, self.cap, C.byref(self.s),
                                                                ptr(self.ws), self.ws_bytes, _lib.stream_ptr()))


def _exact_bins(n: int, gm_s, tile_count: torch.Tensor, H: int, W: int, ranges: torch.Tensor, num_rendered: torch.Tensor,
                region_count: torch.Tensor):
    """Bins of k views at exactly their duplicate counts, the sums of the per-tile counts preprocess wrote into tile_count
    [k, tiles + 1] (gm_s[j]: the RdgGeom of view j), read in ONE host read for all k.  View j is binned (rdg_bin_tiles) in
    buffers of max(count, 1) when the generator reaches it, so that the k views' buffers are not all alive at once.  Nothing
    overflows or is re-binned, and the duplicate-capacity state (_capacity, a pending sync-free count) is neither read nor
    changed."""
    counts = tile_count[:, :tiles_of(H, W)].sum(1).tolist()
    for j, d in enumerate(counts):
        bins = Bins(n, H, W, max(int(d), 1), ranges, num_rendered, region_count)
        bins.bin(gm_s[j])
        yield bins


def _blend_bwd_scratch(n: int, dev: torch.device) -> Optional[torch.Tensor]:
    """rdg_blend_bwd_deterministic's scratch for n Gaussians under config.deterministic, else None."""
    if not config.deterministic:
        return None
    return torch.empty(max(int(_lib.load().rdg_blend_bwd_deterministic_scratch_bytes(n)), 8), dtype=torch.uint8, device=dev)


def _blend_bwd(n: int, gm_s: RdgGeom, bins_s: RdgBins, vw_s: RdgView, img_s: RdgImage, dL_dcolor, dL_ddepth, dL_dalpha,
               acc: torch.Tensor, scratch: Optional[torch.Tensor] = None):
    """The blend backward into acc [n, NACC]: rdg_blend_bwd, or under config.deterministic rdg_blend_bwd_deterministic, with
    the "deterministic" tunable (which also puts the per-Gaussian backward on one CTA) set to match.  scratch: from
    _blend_bwd_scratch; allocated here when None, so a caller that captures a CUDA graph passes its own."""
    lib, stream = _lib.load(), _lib.stream_ptr()
    _lib.set_tunable("deterministic", 1 if config.deterministic else 0)
    args = (n, C.byref(gm_s), C.byref(bins_s), C.byref(vw_s), C.byref(img_s), ptr(dL_dcolor), ptr(dL_ddepth), ptr(dL_dalpha),
            ptr(acc))
    if config.deterministic:
        if scratch is None:
            scratch = _blend_bwd_scratch(n, acc.device)
        check(lib.rdg_blend_bwd_deterministic(*args, ptr(scratch), scratch.numel(), stream))
    else:
        check(lib.rdg_blend_bwd(*args, stream))


def per_view(fn: str, name: str, value, n: int) -> List[float]:
    """A float, or one float per view, as a list of n floats; ValueError prefixed with the caller fn otherwise."""
    vals = [float(t) for t in value] if hasattr(value, "__len__") else [float(value)] * n
    if len(vals) != n:
        raise ValueError(f"{fn}: {name} must be a float or {n} values, got {len(vals)}")
    return vals


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
    ntiles = tiles_of(H, W)
    f32 = dict(dtype=torch.float32, device=dev)
    use_tiles = config.binning == "tiles" and not config.debug_keep_unsorted
    geom = _alloc_geom(n, dev, tile_count=torch.empty(ntiles + 1, dtype=torch.int32, device=dev) if use_tiles else None)
    if config.debug_activated:
        geom["dbg_activated"] = torch.zeros(n, 11, **f32)
    sc_s, vw_s, gm_s = _scene_struct(scene), _view_struct(view), _geom_struct(geom)
    check(lib.rdg_preprocess_fwd(C.byref(sc_s), C.byref(vw_s), C.byref(gm_s), stream))
    if stage_hook:
        stage_hook("preprocess_fwd")

    st = _cap_state(dev, n)
    if not config.capturing:
        _check_pending(st)
    ranges = torch.empty(ntiles, 2, dtype=torch.int32, device=dev)
    point_offsets = torch.empty(n, dtype=torch.int32, device=dev)
    num_rendered = torch.empty(2, dtype=torch.int32, device=dev)
    region_count = torch.empty(2 * ntiles, dtype=torch.int32, device=dev)
    while True:
        bins = Bins(n, H, W, int(st["cap"]), ranges, num_rendered, region_count, keys=config.emit_sorted_keys,
                    lsd=not use_tiles, point_offsets=point_offsets)
        bins.bin(gm_s)
        if config.sync_free:
            # (under graph capture the pinned buffer was allocated beforehand: no cudaHostAlloc inside a capture)
            host = config.capture_host if config.capturing else torch.empty(2, dtype=torch.int32, pin_memory=True)
            host.copy_(num_rendered, non_blocking=True)
            ev = None
            if not config.capturing:
                ev = torch.cuda.Event()
                ev.record()
            st["pending"] = (host, ev, bins.cap)
            break
        d = int(num_rendered[0].item())          # the reference's one host read per forward
        if d <= bins.cap:
            if d * config.headroom > bins.cap:
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
    img = _image_struct(color, depth, alpha, final_T, n_contrib)
    check(lib.rdg_blend_fwd(n, C.byref(gm_s), C.byref(bins.s), C.byref(vw_s), C.byref(img), stream))
    if stage_hook:
        stage_hook("blend_fwd")

    extras = {"keys_sorted": bins.keys, "point_offsets": point_offsets, "region_ids": bins.region_ids,
              "region_masks": bins.region_masks, "region_count": region_count}
    if config.debug_keep_unsorted:
        extras["keys_unsorted"], extras["vals_unsorted"] = bins.keys_unsorted, bins.vals_unsorted
    state = FwdState(scene=scene, view=view, n=n, geom=geom, vals_sorted=bins.vals, ranges=ranges,
                     num_rendered=num_rendered, final_T=final_T, n_contrib=n_contrib, d_cap=bins.cap, extras=extras,
                     bins=bins.s)
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
        geoms = [_alloc_geom(n, dev, radii=radii[lo + j], tile_count=tile_count[j]) for j in range(k)]
        vw_s = (RdgView * k)(*[_view_struct(v) for v in pv])
        gm_s = (RdgGeom * k)(*[_geom_struct(g) for g in geoms])
        bts = None if basis_ts is None else basis_ts[lo:lo + k].contiguous()
        check(lib.rdg_preprocess_fwd_views(C.byref(sc_s), ptr(bts), k, vw_s, gm_s, stream))
        if stage_hook:
            stage_hook("preprocess_fwd")
        for j, bins in enumerate(_exact_bins(n, gm_s, tile_count, H, W, ranges, num_rendered, region_count)):
            v = lo + j
            img = _image_struct(color[v], depth[v], alpha[v], final_T, n_contrib)
            check(lib.rdg_blend_fwd(n, C.byref(gm_s[j]), C.byref(bins.s), C.byref(vw_s[j]), C.byref(img), stream))
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
    # (tile_count zeroed here as well: without Gaussians preprocess returns before it zeroes it)
    tile_count = torch.zeros(1, ntiles + 1, dtype=torch.int32, device=dev)
    geom = _alloc_geom(n, dev, tile_count=tile_count[0])
    sc_s, gm_s = _scene_struct(scene), _geom_struct(geom)
    sc_s.basis_t = ptr(basis_t_src) if sc_s.use_deform else None
    check(lib.rdg_preprocess_fwd(C.byref(sc_s), C.byref(_view_struct(view_src)), C.byref(gm_s), stream))
    sc_s.basis_t = None                                          # rdg_track_attrs takes B(t_m) on its own
    ranges = torch.empty(ntiles, 2, dtype=torch.int32, device=dev)
    num_rendered = torch.empty(2, dtype=torch.int32, device=dev)
    region_count = torch.empty(2 * ntiles, dtype=torch.int32, device=dev)
    (bins,) = _exact_bins(n, [gm_s], tile_count, H, W, ranges, num_rendered, region_count)
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
            img = _image_struct(S[j], blend_depth, alpha, final_T, n_contrib)
            check(lib.rdg_blend_fwd(n, C.byref(gm_s), C.byref(bins.s), C.byref(vw_blend), C.byref(img), stream))
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


RECORD_FLOATS = 62   # RDG_3DGS_RECORD_FLOATS: x y z nx ny nz f_dc_0..2 f_rest_0..44 opacity scale_0..2 rot_0..3


def export_3dgs(scene: SceneArgs, sh_degree: int, device: torch.device) -> torch.Tensor:
    """The scene at B(t) = scene.basis_t as 3DGS PLY vertex records [N, 62] float32 on the device, static rows first
    (rdg_export_3dgs, INTEGRATION.md §11).  scene: raw parameters, no colors_precomp.  One launch, no host read."""
    ns, nd = scene.counts()
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("rodygs_b200 runs on CUDA tensors only (no CPU fallback)")
    records = torch.empty(ns + nd, RECORD_FLOATS, dtype=torch.float32, device=dev)
    sc = _scene_struct(scene)
    check(_lib.load().rdg_export_3dgs(C.byref(sc), int(sh_degree), ptr(records), _lib.stream_ptr()))
    return records


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
    img = _image_struct(None, None, None, state.final_T, state.n_contrib)

    def c(t):
        return None if t is None else t.contiguous()

    dL_dcolor, dL_ddepth, dL_dalpha = c(dL_dcolor), c(dL_ddepth), c(dL_dalpha)
    _blend_bwd(n, gm_s, state.bins, vw_s, img, dL_dcolor, dL_ddepth, dL_dalpha, acc)
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
