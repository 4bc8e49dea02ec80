"""Rendering batches of views (rdg_preprocess_fwd_views, engine.render_views, SplatTrainStep.render_views).

The yardstick is the single-view path: every output of a batched render must be bit-identical to engine.render_forward of
the same scene and view, and the batched preprocess to rdg_preprocess_fwd, at every SH degree, with and without the staged
motion table, for static, dynamic and mixed scenes, at ragged image sizes and with Gaussians behind the near plane (the
synthetic scenes put 1 % there)."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import pytest
import torch

from test_checkpoint import _cpu_step
from test_gpu_metrics import _same, _snapshot

# largest T whose table rows the batched kernel stages in shared memory (RDG_VIEWS_TABLE_MAX in preprocess_fwd.cu)
TABLE_SMEM_MAX = 137


# ================================================================ CPU ==

def _abi_args(nv=2, n_static=4):
    from rodygs_b200 import _lib
    mat = (C.c_float * 16)()
    scene = _lib.RdgScene()
    scene.n_static = n_static
    views = (_lib.RdgView * 9)()
    for v in views:
        v.height, v.width, v.sh_degree, v.scale_modifier = 32, 48, 3, 1.0
        v.tanfovx = v.tanfovy = 0.5
        v.viewmatrix = v.projmatrix = C.addressof(mat)
    geoms = (_lib.RdgGeom * 9)()
    return scene, views, geoms, mat


def test_abi_refuses_bad_arguments_without_a_gpu():
    from rodygs_b200 import _lib
    lib = _lib.load()
    scene, views, geoms, mat = _abi_args()

    def call(nv=2, sc=scene, vw=views, gm=geoms, bts=None):
        return lib.rdg_preprocess_fwd_views(None if sc is None else C.byref(sc), bts, nv, vw, gm, None)

    for nv in (0, -1, 9):
        assert call(nv) == -1 and b"num_views" in lib.rdg_last_error(), nv
    assert call(sc=None) == -1 and b"null argument" in lib.rdg_last_error()
    assert call(vw=None) == -1 and b"null argument" in lib.rdg_last_error()
    assert call(gm=None) == -1 and b"null argument" in lib.rdg_last_error()
    for field, value in (("height", 33), ("width", 47), ("sh_degree", 2), ("scale_modifier", 0.5)):
        _, vw, _, _ = _abi_args()
        setattr(vw[1], field, value)
        assert call(vw=vw) == -1 and b"must share" in lib.rdg_last_error(), field
        assert call(nv=1, vw=vw) == -1 and b"null geometry buffer" in lib.rdg_last_error(), field   # one view: nothing to share
    _, vw, _, _ = _abi_args()
    vw[1].projmatrix = None
    assert call(vw=vw) == -1 and b"null camera matrix" in lib.rdg_last_error()
    vw[1].projmatrix, vw[1].sh_degree = C.addressof(mat), 4
    assert call(vw=vw) == -1 and b"sh_degree" in lib.rdg_last_error()
    sc, _, _, _ = _abi_args()
    sc.basis_t = C.addressof(mat)
    assert call(sc=sc) == -1 and b"basis_t must be NULL" in lib.rdg_last_error()
    assert call() == -1 and b"null geometry buffer" in lib.rdg_last_error()
    buf = (C.c_float * 64)()
    for g in geoms:
        g.radii = g.tiles_touched = g.p0 = g.p1 = g.p2 = g.clamped = C.addressof(buf)
    assert call() == -1 and b"null static parameter" in lib.rdg_last_error()
    sc, _, _, _ = _abi_args(n_static=0)
    sc.n_dynamic, sc.raw, sc.use_deform, sc.num_basis, sc.num_times = 4, 1, 1, 16, 5
    sc.dy.xyz = sc.dy.scaling = sc.dy.rotation = sc.dy.opacity = sc.dy.sh_dc = sc.dy.sh_rest = C.addressof(buf)
    sc.motion_coeff = sc.time_ind = sc.table = C.addressof(buf)
    assert call(sc=sc) == -1 and b"null deformation input" in lib.rdg_last_error()      # basis_ts missing
    sc.n_dynamic = 0
    assert call(sc=sc) == 0                                                                # nothing to do: no launch


def test_render_views_checks_its_arguments_on_the_host():
    step = _cpu_step(n=50)
    V = 3
    vm, pm, bts = torch.eye(4).repeat(V, 1, 1), torch.eye(4).repeat(V, 1, 1), torch.zeros(V, 16, 7)
    with pytest.raises(ValueError, match="V >= 1"):
        step.render_views(torch.zeros(0, 4, 4), pm, 0.5, 0.5, bts)
    with pytest.raises(ValueError, match="V >= 1"):
        step.render_views(None, pm, 0.5, 0.5, bts)
    with pytest.raises(ValueError, match="projmats must be"):
        step.render_views(vm, pm[:2], 0.5, 0.5, bts)
    with pytest.raises(ValueError, match="viewmats must be"):
        step.render_views(vm.double(), pm, 0.5, 0.5, bts)
    with pytest.raises(ValueError, match="basis_ts must be"):
        step.render_views(vm, pm, 0.5, 0.5, bts[:, :8])
    with pytest.raises(ValueError, match="basis_ts must be"):
        step.render_views(vm, pm, 0.5, 0.5, None)
    with pytest.raises(ValueError, match="tanfovx must be a float or 3 values, got 2"):
        step.render_views(vm, pm, [0.5, 0.5], 0.5, bts)
    with pytest.raises(ValueError, match="tanfovy must be a float or 3 values, got 4"):
        step.render_views(vm, pm, 0.5, [0.5] * 4, bts)


def _compile_preprocess(tmp):
    from rodygs_b200 import build
    obj = os.path.join(tmp, "preprocess_fwd.o")
    r = subprocess.run([build._nvcc(), *build.ARCH, *build.COMMON, *build.SOURCES["preprocess_fwd.cu"], "-Xptxas", "-v", "-c",
                        os.path.join(build.CSRC, "preprocess_fwd.cu"), "-o", obj], capture_output=True, text=True, check=True)
    return r.stderr, obj


def test_batched_kernel_does_not_spill():
    """`-Xptxas -v` for every instantiation of the batched kernel: no spills at the 128 registers that 2 CTAs per SM allow.
    The 144-byte stack frame of the RAW instantiations is the one the single-view kernel has too (the coefficient array
    indexed at run time when num_basis < 16)."""
    with tempfile.TemporaryDirectory() as tmp:
        log, _ = _compile_preprocess(tmp)
    info, regs, name = {}, {}, None
    for line in log.splitlines():
        hit = re.search(r"Compiling entry function '(\w+)'", line)
        if hit:
            name = hit.group(1)
        elif name and "spill" in line:
            info[name] = line.strip()
        elif name and "Used" in line:
            regs[name] = int(re.search(r"Used (\d+) registers", line).group(1))
    new = [n for n in info if "preprocess_fwd_views_kernel" in n]
    assert len(new) == 8, sorted(info)
    for n in new:
        assert "0 bytes spill stores, 0 bytes spill loads" in info[n], (n, info[n])
        assert regs[n] <= 128, (n, regs[n])


# ================================================================ GPU ==

def _make_step(N, H, W, T=6, sh_degree=3, dynamic_fraction=0.5, seed=3):
    from rodygs_b200 import synthetic
    from rodygs_b200.trainer import SplatTrainStep
    scene = synthetic.to_device(synthetic.make_scene(N, H, W, T, seed=seed, dynamic_fraction=dynamic_fraction), "cuda")
    return SplatTrainStep(scene, H, W, sh_degree=sh_degree, w_pearson=0.0)


def _views(step, V, seed=0):
    """V cameras around the scene with per-view tanfov and B(t) = a table row plus noise (a time between the frames)."""
    from rodygs_b200 import synthetic
    cams = [synthetic.make_camera(v, max(V, 2), step.H, step.W, step.T) for v in range(V)]
    vms = torch.stack([c.world_view_transform.t().contiguous() for c in cams]).cuda()
    pms = torch.stack([c.projection_matrix.t().contiguous() for c in cams]).cuda()
    g = torch.Generator(device="cuda").manual_seed(seed)
    bts = torch.stack([step.p("table")[c.time_index] for c in cams])
    bts = (bts + 0.01 * torch.randn(bts.shape, device="cuda", generator=g)).contiguous()
    fx = [c.tanfovx * (1.0 + 0.03 * v) for v, c in enumerate(cams)]
    fy = [c.tanfovy * (1.0 - 0.02 * v) for v, c in enumerate(cams)]
    return vms, pms, fx, fy, bts


def _reference(step, vms, pms, fx, fy, bts):
    from rodygs_b200 import engine
    out = []
    for v in range(vms.shape[0]):
        scene, view = step._scene_view(vms[v], pms[v], fx[v], fy[v], bts[v] if step.nd > 0 else None)
        out.append(engine.render_forward(scene, view, keep_for_backward=False)[:4])
    return [torch.stack([o[k] for o in out]) for k in range(4)]


def _assert_identical(step, V, seed=0):
    vms, pms, fx, fy, bts = _views(step, V, seed)
    got = step.render_views(vms, pms, fx, fy, bts if step.nd > 0 else None)
    ref = _reference(step, vms, pms, fx, fy, bts)
    for name, a, b in zip(("color", "depth", "alpha", "radii"), got, ref):
        assert a.shape == b.shape and a.dtype == b.dtype, name
        assert torch.equal(a, b), (name, (a != b).sum().item())
    assert (got[3] > 0).any() and (got[3] == 0).any()       # something visible, something culled
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("sh_degree", [0, 1, 2, 3])
@pytest.mark.parametrize("T", [6, TABLE_SMEM_MAX, TABLE_SMEM_MAX + 1])
def test_mixed_scene_every_degree_both_table_paths(sh_degree, T):
    _assert_identical(_make_step(20_000, 176, 208, T=T, sh_degree=sh_degree), 8)


@pytest.mark.gpu
@pytest.mark.parametrize("dynamic_fraction", [0.0, 1.0])
@pytest.mark.parametrize("T", [6, 150])
def test_static_only_and_dynamic_only_scenes(dynamic_fraction, T):
    _assert_identical(_make_step(20_000, 176, 208, T=T, dynamic_fraction=dynamic_fraction), 3)


@pytest.mark.gpu
@pytest.mark.parametrize("V", [1, 3, 8, 11])
def test_view_counts_and_two_passes_at_a_ragged_size(V):
    """97x131: neither side a multiple of the 16-pixel tile.  11 views: a pass of 8 and a pass of 3."""
    _assert_identical(_make_step(30_000, 97, 131, T=12), V, seed=V)


@pytest.mark.gpu
def test_odd_chunk_sizes_and_the_copy_path():
    """Model sizes that are not multiples of the 256-Gaussian chunk (the SH rows of the last chunks are copied by the threads,
    not the bulk copy) and more chunks than CTAs."""
    _assert_identical(_make_step(300_001, 176, 208, T=40, seed=9), 5)


@pytest.mark.gpu
def test_entry_point_matches_single_view_preprocess_with_differing_backgrounds():
    """rdg_preprocess_fwd_views against rdg_preprocess_fwd view by view, every geometry output including the tile counts and
    the activated parameters; then the blends of views that differ in bg as well."""
    from rodygs_b200 import _lib, engine
    lib = _lib.load()
    step = _make_step(20_000, 176, 208, T=6)
    V = 4
    vms, pms, fx, fy, bts = _views(step, V, seed=11)
    n = step.ns + step.nd
    tiles = engine.tiles_of(step.H, step.W)

    def geom():
        f32 = dict(dtype=torch.float32, device="cuda")
        return {"radii": torch.zeros(n, dtype=torch.int32, device="cuda"), "tiles_touched": torch.zeros(n, dtype=torch.int32, device="cuda"),
                "p0": torch.zeros(n, 4, **f32), "p1": torch.zeros(n, 4, **f32), "p2": torch.zeros(n, 2, **f32),
                "clamped": torch.zeros(n, dtype=torch.uint8, device="cuda"), "dbg_activated": torch.zeros(n, 11, **f32),
                "tile_count": torch.full((tiles + 1,), 7, dtype=torch.int32, device="cuda")}

    bgs = torch.rand(V, 3, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    scenes_views = [step._scene_view(vms[v], pms[v], fx[v], fy[v], bts[v]) for v in range(V)]
    views = []
    for v, (_, view) in enumerate(scenes_views):
        view.bg = bgs[v]
        views.append(view)
    batched = [geom() for _ in range(V)]
    scene = scenes_views[0][0]
    scene.basis_t = None
    sc_s = engine._scene_struct(scene)
    vw_s = (_lib.RdgView * V)(*[engine._view_struct(w) for w in views])
    gm_s = (_lib.RdgGeom * V)(*[engine._geom_struct(g) for g in batched])
    _lib.check(lib.rdg_preprocess_fwd_views(C.byref(sc_s), bts.data_ptr(), V, vw_s, gm_s, _lib.stream_ptr()))
    for v in range(V):
        single = geom()
        sc1, vw1 = step._scene_view(vms[v], pms[v], fx[v], fy[v], bts[v])
        _lib.check(lib.rdg_preprocess_fwd(C.byref(engine._scene_struct(sc1)), C.byref(engine._view_struct(vw1)),
                                          C.byref(engine._geom_struct(single)), _lib.stream_ptr()))
        for k in single:
            assert torch.equal(single[k], batched[v][k]), (v, k)
    ref = []
    for v in range(V):
        sc1, vw1 = step._scene_view(vms[v], pms[v], fx[v], fy[v], bts[v])
        vw1.bg = bgs[v]
        ref.append(engine.render_forward(sc1, vw1, keep_for_backward=False)[:4])
    got = engine.render_views(scene, views, bts)
    for k in range(4):
        assert torch.equal(got[k], torch.stack([r[k] for r in ref])), k
    assert not torch.equal(got[0][0], got[0][1])


def _camera_snapshot(step):
    return {k: (v.clone() if torch.is_tensor(v) else v) for k, v in step.cameras.items()}


@pytest.mark.gpu
def test_render_views_leaves_the_training_state_alone():
    """After forward_backward (+ exchange_grads(defer_sh=True)), densification statistics, both optimisers and a camera table:
    every piece of training state is bit-identical after render_views, the objects the next calls read are the same
    objects, the duplicate capacity is untouched, and two calls return the same bits."""
    from rodygs_b200 import engine
    from rodygs_b200.optim import CameraLRs, GaussianLRs
    step = _make_step(20_000, 176, 208)
    step.attach_optimizer("static", GaussianLRs())
    step.attach_optimizer("dynamic", GaussianLRs(scaling_lr=0.001, motion_coeff_lr=1.6e-4))
    step.enable_densification("static")
    step.enable_densification("dynamic")
    step.enable_factored_exchange(views_per_rank=1, world_size=1)
    vms, pms, fx, fy, bts = _views(step, 9)
    step.enable_camera_learning(vms[:2].contiguous(), CameraLRs(1e-4, 1e-4))
    gt = torch.rand(3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    for it in (1, 2):
        step.forward_backward(vms[0], pms[0], fx[0], fy[0], bts[0], gt, None, dcolor_slot=0)
        step.exchange_grads(vms[:1].contiguous(), bts[:1].contiguous(), defer_sh=True)
        if it == 1:
            for tag in ("static", "dynamic"):
                step.add_densification_stats(tag)
                step.optimizer_step(tag, it)
    torch.cuda.synchronize()
    before, cams = _snapshot(step), _camera_snapshot(step)
    cap = {k: dict(v) for k, v in engine._capacity.items()}
    first = step.render_views(vms, pms, fx, fy, bts)
    second = step.render_views(vms, pms, fx, fy, bts)
    torch.cuda.synchronize()
    after = _snapshot(step)
    assert all(torch.equal(a, b) for a, b in zip(first, second))
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
    """Under config.sync_free the training step leaves its duplicate count unread.  render_views neither reads nor clears
    it: here the pending record claims buffers far smaller than the frame needed, render_views still renders (and the
    same bits as without a pending count), and the next forward_backward raises the overflow that belongs to it."""
    from rodygs_b200 import engine
    step = _make_step(20_000, 176, 208)
    vms, pms, fx, fy, bts = _views(step, 3)
    ref = step.render_views(vms, pms, fx, fy, bts)
    gt = torch.rand(3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(6))
    saved = engine.config.sync_free
    engine.config.sync_free = True
    try:
        step.forward_backward(vms[0], pms[0], fx[0], fy[0], bts[0], gt, None)
        st = engine._cap_state(step.params.device, step.ns + step.nd)
        host, ev, _ = st["pending"]
        st["pending"] = pending = (host, ev, 1)          # as if that frame had been truncated
        cap = st["cap"]
        got = step.render_views(vms, pms, fx, fy, bts)
        assert st["pending"] is pending and st["cap"] == cap
        assert all(torch.equal(a, b) for a, b in zip(got, ref))
        with pytest.raises(RuntimeError, match="truncated"):
            step.forward_backward(vms[0], pms[0], fx[0], fy[0], bts[0], gt, None)
    finally:
        engine.config.sync_free = saved
        engine._cap_state(step.params.device, step.ns + step.nd)["pending"] = None
