"""Test-time pose refinement (rdg_pose_adam, rdg_l2_loss, rodygs_b200.pose.refine_poses, SplatTrainStep.refine_poses).

The references: a float64 torch restatement of V(q, T) (tools/pose_refine_bench.view_from_pose) with autograd for the
chain rule, torch.optim.Adam for the update, float64 torch for the loss, and the reference-shaped loop (drop-in
GaussianRasterizer + the same V(q, T) with autograd + L2 + torch.optim.Adam) for whole iterations."""
import ctypes as C
import importlib.util
import math
import os

import numpy as np
import pytest
import torch

from conftest import ROOT
from test_gpu_metrics import _make_step, _same, _snapshot, _views

_spec = importlib.util.spec_from_file_location("pose_refine_bench", os.path.join(ROOT, "tools", "pose_refine_bench.py"))
bench = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(bench)


# ================================================================ CPU ==

def test_struct_layout_matches_header():
    from rodygs_b200 import _lib
    assert C.sizeof(_lib.RdgPoseAdam) == 9 * 8 + 4 * 8 + 2 * 4


def test_abi_refuses_bad_arguments_without_a_gpu():
    from rodygs_b200 import _lib
    lib = _lib.load()
    buf = (C.c_float * 64)()
    a = _lib.RdgPoseAdam(param=C.addressof(buf), exp_avg=C.addressof(buf), exp_avg_sq=C.addressof(buf), step=C.addressof(buf),
                         dL_dV=C.addressof(buf), viewmatrix=C.addressof(buf), lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8,
                         max_steps=10)
    assert lib.rdg_pose_adam(None, 1, None) == -1 and b"args" in lib.rdg_last_error()
    for field in ("param", "viewmatrix", "exp_avg", "exp_avg_sq", "step", "dL_dV"):
        b = _lib.RdgPoseAdam.from_buffer_copy(a)
        setattr(b, field, None)
        assert lib.rdg_pose_adam(C.byref(b), 1, None) == -1
        assert field.encode() in lib.rdg_last_error(), field
    for field, value in (("max_steps", 0), ("lr", 0.0), ("lr", float("nan")), ("beta1", 1.0), ("beta2", -0.1), ("eps", -1.0)):
        b = _lib.RdgPoseAdam.from_buffer_copy(a)
        setattr(b, field, value)
        assert lib.rdg_pose_adam(C.byref(b), 1, None) == -1
        assert field.encode() in lib.rdg_last_error(), field
    b = _lib.RdgPoseAdam.from_buffer_copy(a)
    b.num_rendered = C.addressof(buf)
    assert lib.rdg_pose_adam(C.byref(b), 1, None) == -1 and b"overflow" in lib.rdg_last_error()
    assert lib.rdg_pose_adam(C.byref(a), 2, None) == -1 and b"update" in lib.rdg_last_error()

    ws = lib.rdg_l2_loss_workspace_bytes(3, 1080, 1920)
    assert ws > 0 and ws % 256 == 0
    for args, word in (((0, 8, 8), b"channels"), ((3, 0, 8), b"height"), ((3, 8, 0), b"width")):
        assert lib.rdg_l2_loss_workspace_bytes(*args) == -1 and word in lib.rdg_last_error()
        assert lib.rdg_l2_loss(buf, buf, *args, buf, 4, buf, buf, buf, 1 << 20, None) == -1 and word in lib.rdg_last_error()
    for i, word in ((0, b"pred"), (1, b"gt"), (2, b"step"), (3, b"history"), (4, b"dL_dpred"), (5, b"workspace")):
        p = [buf] * 6
        p[i] = None
        assert lib.rdg_l2_loss(p[0], p[1], 3, 8, 8, p[2], 4, p[3], p[4], p[5], 1 << 20, None) == -1
        assert word in lib.rdg_last_error(), word
    assert lib.rdg_l2_loss(buf, buf, 3, 8, 8, buf, 0, buf, buf, buf, 1 << 20, None) == -1 and b"max_steps" in lib.rdg_last_error()
    small = lib.rdg_l2_loss_workspace_bytes(3, 8, 8)
    assert lib.rdg_l2_loss(buf, buf, 3, 8, 8, buf, 4, buf, buf, buf, small - 1, None) == -1
    assert b"workspace_bytes" in lib.rdg_last_error()


def _cpu_args(n=10, H=8, W=12, V=2, dev="cpu"):
    g = torch.Generator().manual_seed(0)
    static = {"xyz": torch.randn(n, 3, generator=g), "features_dc": torch.randn(n, 1, 3, generator=g),
              "features_rest": torch.zeros(n, 15, 3), "scaling": torch.zeros(n, 3), "rotation": torch.randn(n, 4, generator=g),
              "opacity": torch.zeros(n, 1)}
    vms = torch.eye(4).repeat(V, 1, 1)
    return dict(static={k: v.to(dev) for k, v in static.items()}, height=H, width=W, sh_degree=3, bg=torch.zeros(3, device=dev),
                viewmats=vms.to(dev), projmats=vms.clone().to(dev), tanfovx=0.5, tanfovy=0.4,
                gts=torch.zeros(V, 3, H, W, device=dev), lr=1e-3, iters=5)


def test_refine_poses_refuses_bad_input_on_cpu():
    from rodygs_b200 import pose
    with pytest.raises(ValueError, match="CUDA"):
        pose.refine_poses(**_cpu_args())


def test_pose_from_viewmatrix_inverts_the_restatement_and_refuses_non_rotations():
    """On the CPU in float64: q, T -> V -> (q, T) for random poses (q_r >= 0 after the sign is fixed), camera.npz's V gives
    its quaternion and T_c2w back, and a scaled, skewed or mirrored rotation block is refused with the view named."""
    from rodygs_b200 import pose
    g = torch.Generator().manual_seed(1)
    qs = torch.nn.functional.normalize(torch.randn(64, 4, generator=g, dtype=torch.float64), dim=-1)
    qs[:4] = torch.tensor([[1.0, 0, 0, 0], [0, 1.0, 0, 0], [0, 0, 1.0, 0], [0, 0, 0, 1.0]], dtype=torch.float64)
    Ts = torch.randn(64, 3, generator=g, dtype=torch.float64)
    vms = torch.stack([bench.view_from_pose(q, T) for q, T in zip(qs, Ts)]).float()
    got = pose.pose_from_viewmatrix(vms).double()
    want_q = torch.where(qs[:, :1] < 0, -qs, qs)
    assert torch.allclose(got[:, :4], want_q, atol=2e-6), (got[:, :4] - want_q).abs().max()
    assert torch.allclose(got[:, 4:], Ts, atol=2e-5 * (1 + Ts.abs().max()))
    cam = np.load(os.path.join(ROOT, "tests", "golden", "camera.npz"))
    p = pose.pose_from_viewmatrix(torch.from_numpy(cam["V"]).t().contiguous()[None])[0]
    q = torch.from_numpy(cam["quat"])
    q = -q if q[0] < 0 else q
    assert torch.allclose(p[:4], q, atol=2e-6) and torch.allclose(p[4:], torch.from_numpy(cam["T_c2w"]), atol=2e-6)
    bad = vms[:3].clone()
    bad[1, :3, :3] *= 1.001
    with pytest.raises(ValueError, match=r"view 1: .*not orthonormal"):
        pose.pose_from_viewmatrix(bad)
    bad = vms[:3].clone()
    bad[2, 0, :3] *= -1
    with pytest.raises(ValueError, match=r"view 2"):
        pose.pose_from_viewmatrix(bad)


# ================================================================ GPU ==

def _lib():
    from rodygs_b200 import _lib as L
    return L, L.load()


class _PoseBufs:
    def __init__(self, param, max_steps=100, lr=1e-3):
        from rodygs_b200._lib import RdgPoseAdam, ptr
        dev = "cuda"
        self.param = param.to(dev, torch.float32).contiguous().clone()
        self.m, self.v = torch.zeros(7, device=dev), torch.zeros(7, device=dev)
        self.step = torch.zeros(1, dtype=torch.int32, device=dev)
        self.dV, self.vm, self.grad = torch.zeros(16, device=dev), torch.zeros(16, device=dev), torch.zeros(7, device=dev)
        self.nr, self.ovf = torch.zeros(2, dtype=torch.int32, device=dev), torch.zeros(2, dtype=torch.int32, device=dev)
        self.args = RdgPoseAdam(param=ptr(self.param), exp_avg=ptr(self.m), exp_avg_sq=ptr(self.v), step=ptr(self.step),
                                dL_dV=ptr(self.dV), viewmatrix=ptr(self.vm), grad=ptr(self.grad), num_rendered=ptr(self.nr),
                                overflow=ptr(self.ovf), lr=lr, beta1=0.9, beta2=0.999, eps=1e-8, max_steps=max_steps)

    def call(self, update):
        L, lib = _lib()
        L.check(lib.rdg_pose_adam(C.byref(self.args), update, L.stream_ptr()))
        torch.cuda.synchronize()


@pytest.mark.gpu
def test_parameterisation_reproduces_camera_npz_and_the_restatement():
    cam = np.load(os.path.join(ROOT, "tests", "golden", "camera.npz"))
    b = _PoseBufs(torch.cat([torch.from_numpy(cam["quat"]), torch.from_numpy(cam["T_c2w"])]))
    b.call(0)
    want = torch.from_numpy(cam["V"]).t().reshape(16)
    assert torch.allclose(b.vm.cpu(), want, rtol=0, atol=2e-6), (b.vm.cpu() - want).abs().max()
    assert int(b.step) == 0 and torch.equal(b.param.cpu()[:4], torch.from_numpy(cam["quat"]))
    g = torch.Generator().manual_seed(2)
    for _ in range(8):
        p = torch.randn(7, generator=g)
        p[:4] *= 0.2 + 3 * torch.rand(1, generator=g)            # non-unit q: normalised inside rot()
        b = _PoseBufs(p)
        b.call(0)
        ref = bench.view_from_pose(b.param.double().cpu()[:4], b.param.double().cpu()[4:]).reshape(16)
        assert torch.allclose(b.vm.double().cpu(), ref, rtol=0, atol=4e-6 * (1 + p[4:].abs().max().item())), (b.vm.cpu() - ref).abs().max()


@pytest.mark.gpu
def test_chain_rule_matches_float64_autograd():
    g = torch.Generator().manual_seed(3)
    for _ in range(16):
        p = torch.randn(7, generator=g)
        p[:4] *= 0.3 + 2 * torch.rand(1, generator=g)
        dV = torch.randn(16, generator=g)
        b = _PoseBufs(p)
        b.dV.copy_(dV)
        b.call(1)
        p64 = p.double().clone().requires_grad_(True)
        (bench.view_from_pose(p64[:4], p64[4:]).reshape(16) * dV.double()).sum().backward()
        ref = p64.grad
        got = b.grad.double().cpu()
        err = (got - ref).abs().max() / ref.abs().max()
        assert err < 1e-5, (got, ref)


@pytest.mark.gpu
def test_adam_matches_torch_and_the_guards_block_the_update():
    g = torch.Generator().manual_seed(4)
    p0 = torch.randn(7, generator=g)
    lr = 3e-3
    b = _PoseBufs(p0, max_steps=12, lr=lr)
    q = p0[:4].cuda().clone().requires_grad_(True)
    T = p0[4:].cuda().clone().requires_grad_(True)
    opt = torch.optim.Adam([q, T], lr=lr)
    for it in range(10):
        b.dV.copy_(torch.randn(16, generator=g))
        b.call(1)
        assert torch.equal(b.dV, torch.zeros_like(b.dV)), it
        assert int(b.step) == it + 1
        q.grad, T.grad = b.grad[:4].clone(), b.grad[4:].clone()
        opt.step()
        ref_p = torch.cat([q.detach(), T.detach()])
        st = [opt.state[t] for t in (q, T)]
        ref_m = torch.cat([s["exp_avg"] for s in st])
        ref_v = torch.cat([s["exp_avg_sq"] for s in st])
        for got, ref, name in ((b.param, ref_p, "param"), (b.m, ref_m, "exp_avg"), (b.v, ref_v, "exp_avg_sq")):
            assert torch.allclose(got, ref, rtol=1e-6, atol=1e-12), (it, name, got, ref)
        ref = bench.view_from_pose(b.param.double().cpu()[:4], b.param.double().cpu()[4:]).reshape(16)
        assert torch.allclose(b.vm.double().cpu(), ref, atol=1e-5)
    # binning overflow: nothing applied, counter and moments kept, dL/dV still zeroed, count latched
    snap = [t.clone() for t in (b.param, b.m, b.v, b.step, b.vm)]
    b.nr.copy_(torch.tensor([12345, 1], dtype=torch.int32))
    b.dV.copy_(torch.randn(16, generator=g))
    b.call(1)
    assert all(torch.equal(x, y) for x, y in zip(snap, (b.param, b.m, b.v, b.step, b.vm)))
    assert torch.equal(b.dV, torch.zeros_like(b.dV)) and b.ovf.tolist() == [1, 12345]
    # max_steps reached: the same
    b.nr.zero_()
    b.ovf.zero_()
    b.step.fill_(12)
    b.dV.copy_(torch.randn(16, generator=g))
    snap = [t.clone() for t in (b.param, b.m, b.v, b.step, b.vm)]
    b.call(1)
    assert all(torch.equal(x, y) for x, y in zip(snap, (b.param, b.m, b.v, b.step, b.vm)))
    assert b.ovf.tolist() == [0, 0] and torch.equal(b.dV, torch.zeros_like(b.dV))


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(1080, 1920), (17, 29), (1, 1), (333, 517)])
def test_l2_loss_matches_float64_and_is_reproducible(H, W):
    L, lib = _lib()
    from rodygs_b200._lib import ptr
    g = torch.Generator(device="cuda").manual_seed(H)
    pred = torch.rand(3, H, W, device="cuda", generator=g)
    gt = (pred + 0.1 * torch.randn(3, H, W, device="cuda", generator=g)).contiguous()
    nb = int(lib.rdg_l2_loss_workspace_bytes(3, H, W))
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    step = torch.tensor([3], dtype=torch.int32, device="cuda")
    outs = []
    for _ in range(2):
        hist = torch.full((5,), -1.0, device="cuda")
        dpred = torch.empty_like(pred)
        L.check(lib.rdg_l2_loss(ptr(pred), ptr(gt), 3, H, W, ptr(step), 5, ptr(hist), ptr(dpred), ptr(ws), nb, L.stream_ptr()))
        outs.append((hist.clone(), dpred.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    hist, dpred = outs[0]
    d = pred.double() - gt.double()
    ref = (d * d).mean().item()
    assert hist[[0, 1, 2, 4]].tolist() == [-1.0] * 4
    assert abs(hist[3].item() - ref) <= 1e-4 * ref, (hist[3].item(), ref)
    gref = 2 * d / d.numel()
    assert ((dpred.double() - gref).abs() <= 1e-3 * gref.abs() + 1e-30).all()
    step.fill_(5)                                           # past the history: the gradient only
    L.check(lib.rdg_l2_loss(ptr(pred), ptr(gt), 3, H, W, ptr(step), 5, ptr(hist), ptr(dpred), ptr(ws), nb, L.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(hist, outs[0][0])


# ---- whole loop ------------------------------------------------------------------------------------------------------

def _rot(axis, deg):
    a = torch.nn.functional.normalize(axis.double(), dim=0)
    K = torch.tensor([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]], dtype=torch.float64)
    t = math.radians(deg)
    return torch.eye(3, dtype=torch.float64) + math.sin(t) * K + (1 - math.cos(t)) * K @ K


def _perturbed(vm_true, axis, deg, shift):
    """glm-storage V of the camera turned by `deg` about `axis` (world frame, about its centre) and moved by `shift`."""
    vm = vm_true.double().cpu()
    R, t = vm[:3, :3], vm[3, :3]                 # R_c2w, -R^T C
    C0 = -(R @ t)
    R1 = _rot(axis, deg) @ R
    C1 = C0 + shift
    out = torch.eye(4, dtype=torch.float64)
    out[:3, :3] = R1
    out[3, :3] = -(C1 @ R1)
    return out.float().contiguous().cuda()


def _scene(n, H, W, radius_px, seed=0):
    from rodygs_b200 import synthetic
    scene = synthetic.to_device(synthetic.make_scene(n, H, W, 4, seed=seed, dynamic_fraction=0.0, radius_px=radius_px), "cuda")
    cam = synthetic.make_camera(0, 1, H, W, 4)
    vm = cam.world_view_transform.t().contiguous().cuda()
    pm = cam.projection_matrix.t().contiguous().cuda()
    return scene, cam, vm, pm


def _render(static, cam, vm, pm):
    """The static model at vm through the drop-in rasterizer (activated parameters), colour not clamped."""
    import torch.nn.functional as F
    from rodygs_b200 import GaussianRasterizationSettings, GaussianRasterizer
    rast = GaussianRasterizer(GaussianRasterizationSettings(cam.height, cam.width, cam.tanfovx, cam.tanfovy,
                                                            torch.zeros(3, device="cuda"), 1.0, pm, 3, False, False, True, True))
    with torch.no_grad():
        return rast(means3D=static["xyz"], means2D=torch.zeros_like(static["xyz"]),
                    shs=torch.cat([static["features_dc"], static["features_rest"]], 1).contiguous(),
                    opacities=torch.sigmoid(static["opacity"]), scales=torch.exp(static["scaling"]),
                    rotations=F.normalize(static["rotation"], dim=-1), viewmatrix=vm)[0].contiguous()


@pytest.fixture
def deterministic():
    from rodygs_b200 import engine
    saved = engine.config.deterministic
    engine.config.deterministic = True
    yield
    engine.config.deterministic = saved


def _setup_small(n=20_000, H=176, W=208):
    scene, cam, vm, pm = _scene(n, H, W, radius_px=12.0, seed=5)
    st = scene["static"]
    gt = _render(st, cam, vm, pm)
    vm0 = _perturbed(vm, torch.tensor([0.3, 1.0, -0.2]), 1.0, torch.tensor([0.04, -0.03, 0.05], dtype=torch.float64))
    return st, cam, vm, pm, gt, vm0


@pytest.mark.gpu
def test_one_iteration_gradient_matches_the_reference_loop():
    from rodygs_b200 import pose
    from rodygs_b200._lib import ptr
    st, cam, vm, pm, gt, vm0 = _setup_small()
    bg = torch.zeros(3, device="cuda")
    p0 = pose.pose_from_viewmatrix(vm0[None])[0].contiguous()
    view = pose.ViewArgs(height=cam.height, width=cam.width, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, scale_modifier=1.0,
                         sh_degree=3, viewmatrix=vm0, projmatrix=pm, bg=bg)
    loop = pose._PoseLoop(pose._static_set(st), view, gt, p0, 1e-3, 1)
    grad = torch.zeros(7, device="cuda")
    loop.adam.grad = ptr(grad)
    loop.run()
    _, _, losses, (gq, gT) = bench.reference_loop(st, cam.height, cam.width, 3, bg, pm, cam.tanfovx, cam.tanfovy, gt, p0, 1e-3, 1)
    for got, ref in ((grad[:4], gq), (grad[4:], gT)):
        assert (got - ref).norm() <= 1e-3 * ref.norm(), (got, ref)
    assert abs(loop.history[0].item() - losses[0].item()) <= 1e-4 * losses[0].item()


# Tolerance of the first iterations against the reference loop: Adam's first step is lr * sign(g) per component and later
# steps are ratios of gradient moments, so a 1e-3 relative gradient difference moves each step by ~1e-3 lr; the two loops
# also round V(q, T), the activations and the loss differently.  2 % of the longest possible path (iterations x lr) leaves a
# factor ~20 above that and still fails a wrong sign, a wrong scale or a skipped update (>= 1 lr).
FIRST_ITERS_TOL = 0.02


@pytest.mark.gpu
def test_first_iterations_track_the_reference_loop(deterministic):
    from rodygs_b200 import pose
    st, cam, vm, pm, gt, vm0 = _setup_small()
    bg = torch.zeros(3, device="cuda")
    lr, iters = 1e-3, 5
    out, losses = pose.refine_poses(st, cam.height, cam.width, 3, bg, vm0[None], pm[None], cam.tanfovx, cam.tanfovy, gt[None],
                                    lr, iters)
    p0 = pose.pose_from_viewmatrix(vm0[None])[0].contiguous()
    q, T, ref_losses, _ = bench.reference_loop(st, cam.height, cam.width, 3, bg, pm, cam.tanfovx, cam.tanfovy, gt, p0, lr, iters)
    got = pose.pose_from_viewmatrix(out)[0]
    ref = torch.cat([q / q.norm(), T])
    assert (got - ref).abs().max() <= FIRST_ITERS_TOL * iters * lr, (got, ref)
    assert torch.allclose(losses[0], ref_losses, rtol=1e-3), (losses, ref_losses)


def _errors(vm, vm_true):
    a, b = vm.double().cpu(), vm_true.double().cpu()
    Ra, Rb = a[:3, :3], b[:3, :3]
    cos = ((Ra @ Rb.t()).trace() - 1) / 2
    rot = math.degrees(math.acos(max(-1.0, min(1.0, cos.item()))))
    Ca, Cb = -(Ra @ a[3, :3]), -(Rb @ b[3, :3])
    return rot, (Ca - Cb).norm().item()


@pytest.mark.gpu
def test_recovers_a_perturbed_pose():
    """100k static Gaussians (make_scene's 4-pixel footprints) at 256x384.  The ground truth is the model rendered at V*; the
    start is V* turned 1.5 degrees about a random axis with the centre moved by 2 % of its distance to the scene centre
    (0, 0, 5).  lr = 1e-3, 1000 iterations.  (With 12-pixel footprints the nearest layer hides the rest of the scene, a
    rotation and a sideways move of the camera give almost the same image, and Adam stalls in that valley.)"""
    from rodygs_b200 import pose
    from rodygs_b200.trainer import SplatTrainStep
    H, W = 256, 384
    scene, cam, vm, pm = _scene(100_000, H, W, radius_px=4.0, seed=7)
    st = scene["static"]
    gt = _render(st, cam, vm, pm)
    g = torch.Generator().manual_seed(11)
    axis = torch.randn(3, generator=g)
    vmd = vm.double().cpu()
    C0 = -(vmd[:3, :3] @ vmd[3, :3])
    dist = (C0 - torch.tensor([0.0, 0.0, 5.0], dtype=torch.float64)).norm().item()
    shift = torch.nn.functional.normalize(torch.randn(3, generator=g, dtype=torch.float64), dim=0) * 0.02 * dist
    vm0 = _perturbed(vm, axis, 1.5, shift)
    rot0, c0 = _errors(vm0, vm)
    out, losses = pose.refine_poses(st, H, W, 3, torch.zeros(3, device="cuda"), vm0[None], pm[None], cam.tanfovx, cam.tanfovy,
                                    gt[None], 1e-3, 1000)
    rot1, c1 = _errors(out[0], vm)
    assert rot1 < 0.1 * rot0 and c1 < 0.1 * c0, (rot0, rot1, c0, c1)
    assert losses[0, -1] < 0.05 * losses[0, 0], (losses[0, 0].item(), losses[0, -1].item())
    step = SplatTrainStep(scene, H, W, sh_degree=3, w_pearson=0.0)
    before = step.evaluate(vm0[None], pm[None], cam.tanfovx, cam.tanfovy, None, gt[None])
    after = step.evaluate(out, pm[None], cam.tanfovx, cam.tanfovy, None, gt[None])
    assert after[0, 1] > before[0, 1], (before, after)


@pytest.mark.gpu
def test_deterministic_runs_are_bit_identical(deterministic):
    from rodygs_b200 import pose
    st, cam, vm, pm, gt, vm0 = _setup_small(n=8_000)
    args = (st, cam.height, cam.width, 3, torch.zeros(3, device="cuda"), vm0[None], pm[None], cam.tanfovx, cam.tanfovy, gt[None],
            1e-3, 30)
    a, b = pose.refine_poses(*args), pose.refine_poses(*args)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def _dup_count(st, cam, vm, pm):
    from rodygs_b200 import engine
    from rodygs_b200.engine import SceneArgs, ViewArgs
    from rodygs_b200 import pose
    view = ViewArgs(height=cam.height, width=cam.width, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, scale_modifier=1.0,
                    sh_degree=3, viewmatrix=vm, projmatrix=pm, bg=torch.zeros(3, device="cuda"))
    saved = dict(engine._capacity)
    try:
        return int(engine.render_forward(SceneArgs(st=pose._static_set(st), raw=True), view)[4].num_rendered[0])
    finally:
        engine._capacity.clear()
        engine._capacity.update(saved)


@pytest.mark.gpu
def test_overflow_grows_the_buffers_and_gives_the_ample_capacity_result(deterministic, monkeypatch):
    """headroom 1.0 sizes the buffers to the start pose's count; the start is turned away from the scene so that it sees
    fewer tile instances than the target, and the loop overflows on its way back."""
    from rodygs_b200 import engine, pose
    st, cam, vm, pm, gt, _ = _setup_small(n=8_000)
    d_true = _dup_count(st, cam, vm, pm)
    starts = [_perturbed(vm, torch.tensor([0.0, 1.0, 0.0]), s * 2.0, torch.zeros(3, dtype=torch.float64)) for s in (1, -1)]
    counts = [_dup_count(st, cam, v, pm) for v in starts]
    vm0 = starts[int(counts[1] < counts[0])]
    assert min(counts) < d_true
    args = (st, cam.height, cam.width, 3, torch.zeros(3, device="cuda"), vm0[None], pm[None], cam.tanfovx, cam.tanfovy, gt[None],
            2e-3, 150)
    ample = pose.refine_poses(*args)
    cap_before = {k: dict(v) for k, v in engine._capacity.items()}
    captures = []
    real = pose._PoseLoop._capture

    def counting(self):
        captures.append(self.cap)
        real(self)

    monkeypatch.setattr(pose._PoseLoop, "_capture", counting)
    monkeypatch.setattr(engine.config, "headroom", 1.0)
    tight = pose.refine_poses(*args)
    assert len(captures) >= 2 and captures[-1] > captures[0], captures
    assert {k: dict(v) for k, v in engine._capacity.items()} == cap_before
    tol = FIRST_ITERS_TOL * 150 * 2e-3
    assert (pose.pose_from_viewmatrix(tight[0]) - pose.pose_from_viewmatrix(ample[0])).abs().max() <= tol
    assert torch.allclose(tight[1], ample[1], rtol=1e-3)


@pytest.mark.gpu
def test_refine_poses_leaves_the_training_state_alone():
    """The scenario of test_evaluate_leaves_the_training_state_alone with refine_poses in place of evaluate."""
    from rodygs_b200.optim import GaussianLRs
    step = _make_step(20_000, 176, 208)
    step.attach_optimizer("static", GaussianLRs())
    step.attach_optimizer("dynamic", GaussianLRs(scaling_lr=0.001, motion_coeff_lr=1.6e-4))
    step.enable_densification("static")
    step.enable_densification("dynamic")
    step.enable_factored_exchange(views_per_rank=1, world_size=1)
    cams, vms, pms, bts = _views(step, 3)
    g = torch.Generator(device="cuda").manual_seed(5)
    gt = torch.rand(3, 176, 208, device="cuda", generator=g)
    gts = torch.rand(3, 3, 176, 208, device="cuda", generator=g)
    for it in (1, 2):
        step.forward_backward(vms[0], pms[0], cams[0].tanfovx, cams[0].tanfovy, bts[0], gt, None, dcolor_slot=0)
        step.exchange_grads(vms[:1].contiguous(), bts[:1].contiguous(), defer_sh=True)
        if it == 1:
            for tag in ("static", "dynamic"):
                step.add_densification_stats(tag)
                step.optimizer_step(tag, it)
    torch.cuda.synchronize()
    before = _snapshot(step)
    from rodygs_b200 import engine
    cap_before = {k: (v["cap"], v["pending"]) for k, v in engine._capacity.items()}
    out, losses = step.refine_poses(vms, pms, cams[0].tanfovx, cams[0].tanfovy, gts, 1e-3, 20)
    torch.cuda.synchronize()
    after = _snapshot(step)
    assert torch.isfinite(out).all() and torch.isfinite(losses).all() and losses.shape == (3, 20)
    assert {k: (v["cap"], v["pending"]) for k, v in engine._capacity.items()} == cap_before
    assert after["last_state"] is before["last_state"] and after["deferred"] is before["deferred"]
    assert all(x is y for x, y in zip(after["last_outputs"], before["last_outputs"]))
    for key in before:
        assert _same(before[key], after[key]), key
    for tag in ("static", "dynamic"):
        step.add_densification_stats(tag)
        step.optimizer_step(tag, 2)
    assert not step._deferred["pending"]


@pytest.mark.gpu
def test_step_refine_poses_validates_its_input():
    step = _make_step(4_000, 64, 96)
    cams, vms, pms, bts = _views(step, 2)
    gts = torch.zeros(2, 3, 64, 96, device="cuda")
    t = (cams[0].tanfovx, cams[0].tanfovy)
    with pytest.raises(ValueError, match="viewmats"):
        step.refine_poses(vms.cpu(), pms, *t, gts, 1e-3)
    with pytest.raises(ValueError, match="gts"):
        step.refine_poses(vms, pms, *t, gts[:, :, :10], 1e-3)
    with pytest.raises(ValueError, match="iters"):
        step.refine_poses(vms, pms, *t, gts, 1e-3, iters=0)
    with pytest.raises(ValueError, match="lr"):
        step.refine_poses(vms, pms, *t, gts, 0.0)
    with pytest.raises(ValueError, match="tanfovx"):
        step.refine_poses(vms, pms, [1.0, 2.0, 3.0], t[1], gts, 1e-3)
    bad = vms.clone()
    bad[1, :3, :3] *= 1.01
    with pytest.raises(ValueError, match="view 1"):
        step.refine_poses(bad, pms, *t, gts, 1e-3)


def _dp_worker(rank, world, port, ret):
    import os as _os
    import torch.distributed as dist
    _os.environ["MASTER_ADDR"] = "127.0.0.1"
    _os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        out, losses = _dp_tables()
        ret.put((rank, out.cpu().numpy(), losses.cpu().numpy()))
    finally:
        dist.destroy_process_group()


def _dp_tables():
    from rodygs_b200 import engine
    engine.config.deterministic = True
    step = _make_step(12_000, 176, 208)
    cams, vms, pms, bts = _views(step, 3)
    gts = torch.rand(3, 3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
    return step.refine_poses(vms, pms, [c.tanfovx for c in cams], [c.tanfovy for c in cams], gts, 1e-3, 15)


@pytest.mark.gpu
def test_refine_poses_on_two_ranks_matches_one_process():
    import socket
    import torch.multiprocessing as mp
    from rodygs_b200 import engine
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([ret.get(timeout=300), ret.get(timeout=300)], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    saved = engine.config.deterministic
    try:
        single = [t.cpu() for t in _dp_tables()]
    finally:
        engine.config.deterministic = saved
    for k in (0, 1):
        a, b = torch.from_numpy(res[0][1 + k]), torch.from_numpy(res[1][1 + k])
        assert torch.equal(a, b)
        assert torch.equal(a, single[k]), (a, single[k])
