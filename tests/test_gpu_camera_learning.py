"""Learning the training cameras (rdg_camera_grad, rdg_camera_adam, rdg_camera_views, SplatTrainStep.enable_camera_learning /
camera_step, the checkpoint and export entries, rodygs_b200.optim.CameraLRs, rodygs_b200.metrics.trajectory_errors).

The references: torch autograd through V(q, T) with torch.optim.Adam for the table, rdg_pose_adam for the shared pull-back,
numpy float64 restatements of the learning-rate schedule and of the trajectory errors."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from test_checkpoint import _cpu_step, cpu_rng  # noqa: F401  (cpu_rng is a fixture)
from test_gpu_metrics import _make_step, _views


# ================================================================ CPU ==

def test_abi_refuses_bad_arguments_without_a_gpu():
    from rodygs_b200 import _lib
    lib = _lib.load()
    buf = (C.c_float * 64)()
    b = C.addressof(buf)
    grad_args = [2, b, b, b, 3, b, b, None]
    for i, word in ((1, b"cam_idx"), (2, b"dL_dV_slots"), (3, b"param"), (5, b"grad"), (6, b"error")):
        a = list(grad_args)
        a[i] = None
        assert lib.rdg_camera_grad(*a) == -1 and word in lib.rdg_last_error(), word
    for i, v, word in ((0, -1, b"n_slots"), (4, 0, b"C"), (4, -3, b"C")):
        a = list(grad_args)
        a[i] = v
        assert lib.rdg_camera_grad(*a) == -1 and word in lib.rdg_last_error(), word
    adam_args = [b, b, b, b, 3, 1, 1e-3, 1e-3, 0.9, 0.999, 1e-15, 1.0, b, None]
    for i, word in ((0, b"param"), (1, b"grad"), (2, b"exp_avg"), (3, b"exp_avg_sq"), (12, b"viewmats")):
        a = list(adam_args)
        a[i] = None
        assert lib.rdg_camera_adam(*a) == -1 and word in lib.rdg_last_error(), word
    for i, v, word in ((4, 0, b"C"), (5, 0, b"step"), (5, -2, b"step"), (6, -1e-3, b"lr_q"), (7, float("nan"), b"lr_T"),
                       (8, 1.0, b"beta1"), (9, -0.1, b"beta2"), (10, -1.0, b"eps"), (11, float("inf"), b"grad_scale")):
        a = list(adam_args)
        a[i] = v
        assert lib.rdg_camera_adam(*a) == -1 and word in lib.rdg_last_error(), word
    assert lib.rdg_camera_views(None, 3, b, None) == -1 and b"param" in lib.rdg_last_error()
    assert lib.rdg_camera_views(b, 3, None, None) == -1 and b"viewmats" in lib.rdg_last_error()
    assert lib.rdg_camera_views(b, 0, b, None) == -1 and b"C" in lib.rdg_last_error()


def _np_factor(it, lr):
    warm = 1.0 if lr.warmup_steps == 0 else np.minimum(1.0, it / lr.warmup_steps)
    p = np.clip((it - lr.warmup_steps) / (lr.max_steps - lr.warmup_steps), 0.0, 1.0)
    return warm * (lr.final_ratio + (1.0 - lr.final_ratio) * 0.5 * (1.0 + np.cos(np.pi * p)))


def test_camera_lrs_follow_the_warmup_cosine_formula():
    from rodygs_b200.optim import CameraLRs
    lr = CameraLRs(1e-3, 4e-3, warmup_steps=100, max_steps=1100, final_ratio=0.05)
    for it in (0, 1, 50, 100, 600, 1100, 5000):
        f = _np_factor(np.float64(it), lr)
        q, T = lr.rates(it)
        assert math.isclose(q, 1e-3 * f, rel_tol=1e-14, abs_tol=0) and math.isclose(T, 4e-3 * f, rel_tol=1e-14, abs_tol=0), it
    assert lr.rates(0) == (0.0, 0.0) and lr.factor(100) == 1.0
    assert math.isclose(lr.factor(600), 0.05 + 0.95 * 0.5, rel_tol=1e-14)
    assert math.isclose(lr.factor(1100), 0.05, rel_tol=1e-14) and lr.factor(5000) == lr.factor(1100)
    const = CameraLRs(2e-3, 3e-3)
    assert all(const.rates(it) == (2e-3, 3e-3) for it in (0, 1, 10, 10_000))
    for kwargs, word in ((dict(lr_q=-1.0, lr_T=1.0), "lr_q"), (dict(lr_q=1.0, lr_T=float("nan")), "lr_T"),
                         (dict(lr_q=1.0, lr_T=1.0, warmup_steps=-1), "warmup_steps"),
                         (dict(lr_q=1.0, lr_T=1.0, warmup_steps=10, max_steps=10), "max_steps"),
                         (dict(lr_q=1.0, lr_T=1.0, final_ratio=-0.5), "final_ratio")):
        with pytest.raises(ValueError, match=word):
            CameraLRs(**kwargs)
    with pytest.raises(TypeError):
        CameraLRs(1e-3)                                      # both rates are required


def _np_trajectory_errors(pred, gt):
    """Float64 numpy restatement: Umeyama Sim(3) of the centres, ATE, then RPE of the aligned poses over consecutive pairs."""
    pred, gt = np.asarray(pred, np.float64), np.asarray(gt, np.float64)
    x, y = pred[:, :3, 3], gt[:, :3, 3]
    n = len(x)
    mx, my = x.mean(0), y.mean(0)
    cov = (y - my).T @ (x - mx) / n
    U, D, Vt = np.linalg.svd(cov)
    S = np.eye(3)
    if np.linalg.det(U) * np.linalg.det(Vt) < 0:
        S[2, 2] = -1
    R = U @ S @ Vt
    s = np.trace(np.diag(D) @ S) / (((x - mx) ** 2).sum() / n)
    t = my - s * R @ mx
    al = pred.copy()
    for i in range(n):
        al[i, :3, :3] = R @ pred[i, :3, :3]
        al[i, :3, 3] = s * R @ x[i] + t
    ate = np.sqrt(np.mean(np.sum((al[:, :3, 3] - y) ** 2, 1)))
    tr, rot = [], []
    for i in range(n - 1):
        rel = np.linalg.inv(np.linalg.inv(gt[i]) @ gt[i + 1]) @ (np.linalg.inv(al[i]) @ al[i + 1])
        tr.append(np.linalg.norm(rel[:3, 3]))
        rot.append(np.degrees(np.arccos(np.clip((np.trace(rel[:3, :3]) - 1) / 2, -1, 1))))
    return ate, np.mean(tr), np.mean(rot)


def _rot(axis, deg, dtype=torch.float64):
    a = torch.nn.functional.normalize(axis.to(dtype), dim=0)
    K = torch.tensor([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]], dtype=dtype)
    th = math.radians(deg)
    return torch.eye(3, dtype=dtype) + math.sin(th) * K + (1 - math.cos(th)) * K @ K


def _random_c2w(n, g):
    out = torch.eye(4, dtype=torch.float64).repeat(n, 1, 1)
    for i in range(n):
        out[i, :3, :3] = _rot(torch.randn(3, generator=g), float(torch.rand(1, generator=g)) * 180)
        out[i, :3, 3] = torch.randn(3, generator=g, dtype=torch.float64)
    return out


def test_trajectory_errors_match_the_numpy_restatement():
    from rodygs_b200.metrics import trajectory_errors
    g = torch.Generator().manual_seed(5)
    gt = _random_c2w(40, g)
    pred = gt.clone()
    for i in range(len(pred)):
        pred[i, :3, :3] = _rot(torch.randn(3, generator=g), 2.0) @ pred[i, :3, :3]
        pred[i, :3, 3] = 1.7 * pred[i, :3, 3] + 0.05 * torch.randn(3, generator=g, dtype=torch.float64) + 0.3
    assert all(t.dtype == torch.float64 and t.dim() == 0 for t in trajectory_errors(pred.float(), gt.float()))
    got = trajectory_errors(pred, gt)
    want = _np_trajectory_errors(pred.numpy(), gt.numpy())
    for a, b in zip(got, want):
        assert math.isclose(float(a), b, rel_tol=1e-9), (float(a), b)
    # a ground truth mapped by a Sim(3) is aligned back exactly
    R, s, t = _rot(torch.randn(3, generator=g), 73.0), 0.37, torch.randn(3, generator=g, dtype=torch.float64)
    sim = gt.clone()
    sim[:, :3, :3] = R @ gt[:, :3, :3]
    sim[:, :3, 3] = s * gt[:, :3, 3] @ R.t() + t
    assert all(float(v) < 1e-9 for v in trajectory_errors(sim, gt)), [float(v) for v in trajectory_errors(sim, gt)]
    # centres on a unit square, offsets eps * (0, 0, +-1) alternating: the Umeyama fit is the identity rotation with scale
    # 1 / (1 + eps^2), and ATE = eps / sqrt(1 + eps^2)
    eps = 0.1
    sq = torch.eye(4, dtype=torch.float64).repeat(4, 1, 1)
    sq[:, :3, 3] = torch.tensor([[1.0, 0, 0], [0, 1, 0], [-1, 0, 0], [0, -1, 0]], dtype=torch.float64)
    off = sq.clone()
    off[:, 2, 3] = torch.tensor([eps, -eps, eps, -eps], dtype=torch.float64)
    ate = float(trajectory_errors(off, sq)[0])
    assert math.isclose(ate, eps / math.sqrt(1 + eps * eps), rel_tol=1e-12), ate
    assert math.isclose(ate, _np_trajectory_errors(off.numpy(), sq.numpy())[0], rel_tol=1e-12)
    with pytest.raises(ValueError, match="C >= 2"):
        trajectory_errors(gt[:1], gt[:1])
    with pytest.raises(ValueError, match="4, 4"):
        trajectory_errors(gt[:, :3], gt[:, :3])


def _cpu_camera_step(monkeypatch, C_=6, n=300, seed=0):
    """A CPU step with a camera table (rdg_camera_views is a device launch: the CPU tests check the host logic only)."""
    from rodygs_b200.optim import CameraLRs
    from rodygs_b200.trainer import SplatTrainStep
    monkeypatch.setattr(SplatTrainStep, "_camera_views", lambda self: None)
    step = _cpu_step(n=n, seed=seed)
    g = torch.Generator().manual_seed(seed + 9)
    c2w = _random_c2w(C_, g)
    step.enable_camera_learning(torch.linalg.inv(c2w).transpose(1, 2).float().contiguous(),
                                CameraLRs(1e-3, 2e-3, warmup_steps=3, max_steps=50, final_ratio=0.1))
    cam = step.cameras
    cam["exp_avg"].copy_(torch.randn(C_, 7, generator=g))
    cam["exp_avg_sq"].copy_(torch.rand(C_, 7, generator=g))
    cam["steps"] = 5
    return step


def test_checkpoint_round_trip_of_the_camera_table(tmp_path, cpu_rng, monkeypatch):
    from rodygs_b200 import checkpoint as ck
    src = _cpu_camera_step(monkeypatch)
    path = tmp_path / "ck.pt"
    src.save(path)
    dst = _cpu_step(n=170, seed=4)
    assert getattr(dst, "cameras", None) is None
    dst.load(path)                                            # a state with cameras enables them
    for k in ("param", "exp_avg", "exp_avg_sq"):
        assert torch.equal(dst.cameras[k], src.cameras[k]), k
    assert dst.cameras["steps"] == 5 and dst.cameras["lrs"] == src.cameras["lrs"] and dst.cameras["pending"] == []
    # a mismatched camera count is refused, naming the field, and the step keeps its table
    other = _cpu_camera_step(monkeypatch, C_=4, seed=2)
    before = other.cameras["param"].clone()
    with pytest.raises(ValueError, match=r"cameras\['param'\] holds 6 cameras .* has 4"):
        other.load_state_dict(torch.load(path, weights_only=True))
    assert torch.equal(other.cameras["param"], before)
    # collected gradients that no camera_step has consumed are not saved silently
    src.cameras["pending"].append(0)
    with pytest.raises(RuntimeError, match="camera_step"):
        src.state_dict()
    src.cameras["pending"].clear()
    # export under the reference's names, import, and enable from the imported dict
    out = ck.export_models(src)
    assert out["cameras"]["R_c2ws_quat"].shape == (6, 4) and out["cameras"]["T_c2ws"].shape == (6, 3)
    scene = ck.import_models(out)
    again = _cpu_step(n=120, seed=6)
    again.enable_camera_learning(scene["cameras"], src.cameras["lrs"])
    assert torch.equal(again.cameras["param"], src.cameras["param"])
    bad = dict(out, cameras={"R_c2ws_quat": out["cameras"]["R_c2ws_quat"], "T_c2ws": out["cameras"]["T_c2ws"][:5]})
    with pytest.raises(ValueError, match="T_c2ws"):
        ck.import_models(bad)
    assert "cameras" not in ck.export_models(_cpu_step(n=50, seed=1))


def test_camera_arguments_are_checked_on_the_host(monkeypatch):
    from rodygs_b200.optim import CameraLRs
    step = _cpu_step(n=50)
    with pytest.raises(RuntimeError, match="not enabled"):
        step.camera_viewmatrix(0)
    with pytest.raises(ValueError, match="CameraLRs"):
        step.enable_camera_learning(torch.eye(4).repeat(2, 1, 1), {"lr_q": 1.0})
    bad = torch.eye(4).repeat(3, 1, 1)
    bad[1, :3, :3] *= 1.01
    with pytest.raises(ValueError, match="view 1"):
        step.enable_camera_learning(bad, CameraLRs(1e-3, 1e-3))
    step = _cpu_camera_step(monkeypatch)
    for c in (-1, 6, 1.5, True):
        with pytest.raises(ValueError, match=r"\[0, 6\)"):
            step.collect_camera_grad(c)
    with pytest.raises(ValueError, match="not both"):
        step.forward_backward(torch.eye(4), torch.eye(4), 0.5, 0.5, None, None, None, camera=0)


# ================================================================ GPU ==

def _glm_views(q, T):
    """[C, 4, 4] glm-storage V(q, T) of every row, differentiable (tools/pose_refine_bench.view_from_pose, batched)."""
    r, x, y, z = (q / q.norm(dim=-1, keepdim=True)).unbind(-1)
    R = torch.stack([torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y)], -1),
                     torch.stack([2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x)], -1),
                     torch.stack([2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], -1)], -2)
    top = torch.cat([R, torch.zeros_like(R[:, :, :1])], -1)
    bottom = torch.cat([-(T.unsqueeze(1) @ R), torch.ones_like(R[:, :1, :1])], -1)
    return torch.cat([top, bottom], 1)


def _close(got, ref, tol=1e-6):
    return (got - ref).abs().max().item() <= tol * ref.abs().max().item()


@pytest.mark.gpu
def test_table_matches_torch_autograd_and_adam():
    """7 cameras, 3 slots per iteration (one camera twice), random dL/dV, 20 iterations of CameraLRs' schedule from it = 0
    (lr 0: moments and step count still advance).  Camera 6 has gradient in the first 5 iterations only: it must keep
    moving afterwards, by the same amount as torch's."""
    from rodygs_b200.optim import CameraLRs
    step = _make_step(2000, 48, 64)
    Cn = 7
    g = torch.Generator().manual_seed(21)
    c2w = _random_c2w(Cn, g)
    lrs = CameraLRs(2e-3, 5e-3, warmup_steps=4, max_steps=20, final_ratio=0.2)
    step.enable_camera_learning(torch.linalg.inv(c2w).transpose(1, 2).float().contiguous().cuda(), lrs)
    cam = step.cameras
    q = torch.nn.Parameter(cam["param"][:, :4].clone())
    T = torch.nn.Parameter(cam["param"][:, 4:].clone())
    opt = torch.optim.Adam([{"params": [q], "lr": 0.0}, {"params": [T], "lr": 0.0}], betas=(0.9, 0.999), eps=1e-15)
    assert torch.allclose(cam["viewmats"], _glm_views(q, T).detach().reshape(Cn, 16), atol=2e-6)
    moved_after = []
    for it in range(20):
        cams = [int(c) for c in torch.randint(0, 6, (2,), generator=g)]
        cams = [cams[0], cams[0], 6] if it < 5 else [cams[0], cams[1], cams[0]]
        dVs = torch.randn(3, 16, generator=g).cuda()
        for c, dV in zip(cams, dVs):
            step.view_grad.copy_(dV.view(4, 4))
            step.collect_camera_grad(c)
        before6 = cam["param"][6].clone()
        lr_q, lr_T = step.camera_step(it)
        opt.param_groups[0]["lr"], opt.param_groups[1]["lr"] = lr_q, lr_T
        opt.zero_grad()
        V = _glm_views(q, T)
        sum((dV.view(4, 4) * V[c]).sum() for c, dV in zip(cams, dVs)).backward()
        opt.step()
        ref = torch.cat([q.detach(), T.detach()], 1)
        st = [opt.state[p] for p in (q, T)]
        assert _close(cam["param"], ref), (it, (cam["param"] - ref).abs().max())
        assert _close(cam["exp_avg"], torch.cat([s["exp_avg"] for s in st], 1)), it
        assert _close(cam["exp_avg_sq"], torch.cat([s["exp_avg_sq"] for s in st], 1)), it
        if it >= 6:
            d = cam["param"][6] - before6
            moved_after.append(d.abs().max().item())
    assert min(moved_after) > 0, moved_after
    assert torch.allclose(cam["viewmats"], _glm_views(q, T).detach().reshape(Cn, 16), atol=2e-6)
    assert cam["steps"] == 20 and cam["pending"] == []


@pytest.mark.gpu
def test_one_slot_gives_the_bits_of_rdg_pose_adam():
    from test_pose_refine import _PoseBufs
    from rodygs_b200 import _lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(22)
    for _ in range(16):
        p = torch.randn(7, generator=g)
        p[:4] *= 0.3 + 2 * torch.rand(1, generator=g)
        dV = torch.randn(16, generator=g)
        b = _PoseBufs(p)
        b.dV.copy_(dV)
        b.call(1)
        param = torch.randn(3, 7, generator=g).cuda()
        param[1] = p.cuda()
        grad = torch.full((3, 7), float("nan"), device="cuda")
        err = torch.full((1,), -5, dtype=torch.int32, device="cuda")
        idx = torch.tensor([1], dtype=torch.int32, device="cuda")
        L.check(lib.rdg_camera_grad(1, L.ptr(idx), L.ptr(dV.cuda()), L.ptr(param), 3, L.ptr(grad), L.ptr(err), L.stream_ptr()))
        torch.cuda.synchronize()
        assert torch.equal(grad[1], b.grad) and torch.equal(grad[0], torch.zeros(7, device="cuda")), (grad, b.grad)
        assert int(err) == 0
    # an index outside [0, C) is reported as 1 + its slot and adds to no row; the other slots still count
    idx = torch.tensor([0, 7, -1, 2], dtype=torch.int32, device="cuda")
    dVs = torch.randn(4, 16, generator=g).cuda()
    grad = torch.full((3, 7), float("nan"), device="cuda")
    L.check(lib.rdg_camera_grad(4, L.ptr(idx), L.ptr(dVs), L.ptr(param), 3, L.ptr(grad), L.ptr(err), L.stream_ptr()))
    torch.cuda.synchronize()
    assert int(err) == 2
    assert torch.isfinite(grad).all() and torch.equal(grad[1], torch.zeros(7, device="cuda"))


@pytest.fixture
def deterministic():
    from rodygs_b200 import engine
    saved = engine.config.deterministic
    engine.config.deterministic = True
    yield
    engine.config.deterministic = saved


def _enabled_step(n=12_000, H=176, W=208, V=4, lrs=None):
    from rodygs_b200.optim import CameraLRs
    step = _make_step(n, H, W)
    cams, vms, pms, bts = _views(step, V)
    step.enable_camera_learning(vms, lrs or CameraLRs(1e-3, 1e-3))
    return step, cams, pms, bts


@pytest.mark.gpu
def test_camera_argument_changes_nothing_else(deterministic):
    step, cams, pms, bts = _enabled_step()
    gt = torch.rand(3, step.H, step.W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    c = 2
    args = (pms[c], cams[c].tanfovx, cams[c].tanfovy, bts[c].contiguous(), gt, None)
    step.forward_backward(None, *args, camera=c)
    a = (step.grads.clone(), step.loss_parts.clone(), step.view_grad.clone())
    assert step.cameras["pending"] == [c] and torch.equal(step.cameras["slots"][0], step.view_grad.view(16))
    step.cameras["pending"].clear()
    step.forward_backward(step.camera_viewmatrix(c), *args)
    assert step.cameras["pending"] == []
    for x, y in zip(a, (step.grads, step.loss_parts, step.view_grad)):
        assert torch.equal(x, y)


def _perturbed_glm(vm_glm, axis, deg, shift):
    V = vm_glm.double().cpu().t()
    c2w = torch.linalg.inv(V)
    c2w[:3, :3] = _rot(axis, deg) @ c2w[:3, :3]
    c2w[:3, 3] += shift
    return torch.linalg.inv(c2w).t().float().contiguous().cuda()


def _c2w_of_table(step):
    return torch.linalg.inv(step.cameras["viewmats"].view(-1, 4, 4).transpose(1, 2).double())


@pytest.mark.gpu
def test_recovers_perturbed_training_cameras():
    """8 cameras of the synthetic ring over make_scene's static + dynamic model (4-pixel footprints, 100k Gaussians at
    256x384); the ground truth is the model rendered at the true cameras.  Every camera is turned 1 degree about a random
    axis and its centre moved by 0.04 (1 % of the 4-unit distance to the scene centre).  The Gaussians stay frozen; the
    cameras learn for 1000 iterations of all 8 views (lr 1e-3 for q and T, cosine to 1 %) under the L1 photometric term.
    The ATE after the Sim(3) alignment must fall by at least 5x.  Observed on an NVIDIA B200: ATE 0.0368 -> 1.04e-6, RPE
    2.0e-6 / 1.9e-4 degrees.  (With the default 0.2 D-SSIM weight the same start stalls on a static-only scene at ATE 0.028, a
    local minimum of the SSIM term; with L1 alone it reaches 2e-6 there too.)"""
    from rodygs_b200 import synthetic
    from rodygs_b200.metrics import trajectory_errors
    from rodygs_b200.optim import CameraLRs
    from rodygs_b200.trainer import SplatTrainStep
    V, iters, H, W = 8, 1000, 256, 384
    scene = synthetic.to_device(synthetic.make_scene(100_000, H, W, 6, seed=7), "cuda")
    step = SplatTrainStep(scene, H, W, sh_degree=3, w_l1=1.0, w_dssim=0.0, w_pearson=0.0)
    cams, vms, pms, bts = _views(step, V, n_views=V)
    gts = []
    for c in range(V):
        step.forward_backward(vms[c], pms[c], cams[c].tanfovx, cams[c].tanfovy, bts[c].contiguous(), None, None,
                              forward_only=True)
        gts.append(step.last_outputs[0].clone())
    g = torch.Generator().manual_seed(31)
    start = torch.stack([_perturbed_glm(vms[c], torch.randn(3, generator=g), 1.0,
                                        0.04 * torch.nn.functional.normalize(torch.randn(3, generator=g, dtype=torch.float64), dim=0))
                         for c in range(V)])
    step.enable_camera_learning(start, CameraLRs(1e-3, 1e-3, warmup_steps=0, max_steps=iters, final_ratio=0.01))
    gt_c2w = torch.linalg.inv(vms.transpose(1, 2).double())
    ate0 = float(trajectory_errors(_c2w_of_table(step), gt_c2w)[0])
    for it in range(iters):
        for c in range(V):
            step.forward_backward(None, pms[c], cams[c].tanfovx, cams[c].tanfovy, bts[c].contiguous(), gts[c], None, camera=c)
        step.camera_step(it)
    ate1, rpe_t, rpe_r = (float(x) for x in trajectory_errors(_c2w_of_table(step), gt_c2w))
    print(f"camera recovery: ATE {ate0:.4g} -> {ate1:.4g} (x{ate0 / ate1:.1f}), RPE {rpe_t:.4g} / {rpe_r:.4g} deg")
    assert ate1 * 5 <= ate0, (ate0, ate1, rpe_t, rpe_r)


def _run(step, cams, pms, bts, gts, its):
    for it in its:
        for c in range(len(gts)):
            step.forward_backward(None, pms[c], cams[c].tanfovx, cams[c].tanfovy, bts[c].contiguous(), gts[c], None, camera=c)
        step.camera_step(it)


@pytest.mark.gpu
def test_resumed_camera_learning_matches_the_uninterrupted_run(deterministic, tmp_path):
    from rodygs_b200.optim import CameraLRs
    from rodygs_b200.trainer import SplatTrainStep
    lrs = CameraLRs(2e-3, 1e-3, warmup_steps=2, max_steps=8, final_ratio=0.3)
    a, cams, pms, bts = _enabled_step(lrs=lrs)
    gts = torch.rand(4, 3, a.H, a.W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4))
    _run(a, cams, pms, bts, gts, range(8))
    b, *_ = _enabled_step(lrs=lrs)
    _run(b, cams, pms, bts, gts, range(4))
    b.save(tmp_path / "mid.pt")
    c = SplatTrainStep.from_state_dict(torch.load(tmp_path / "mid.pt", weights_only=True))
    _run(c, cams, pms, bts, gts, range(4, 8))
    for k in ("param", "exp_avg", "exp_avg_sq", "viewmats"):
        assert torch.equal(a.cameras[k], c.cameras[k]), k
    assert a.cameras["steps"] == c.cameras["steps"] == 8


def _dp_cameras(rank, world):
    """Rank r renders view r of camera 1 (views at two times); one process renders both.  Three iterations."""
    step, cams, pms, bts = _enabled_step(V=2)
    gts = torch.rand(2, 3, step.H, step.W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(6))
    mine = [rank] if world > 1 else [0, 1]
    for it in range(3):
        for v in mine:
            step.forward_backward(None, pms[1], cams[1].tanfovx, cams[1].tanfovy, bts[v].contiguous(), gts[v], None, camera=1)
        step.camera_step(it + 1)
    return torch.cat([step.cameras[k] for k in ("param", "exp_avg", "exp_avg_sq")], 1)


def _dp_worker(rank, world, port, ret):
    """Two gloo ranks, on two GPUs when there are two, else both on one."""
    import os
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank % torch.cuda.device_count())
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ret.put((rank, _dp_cameras(rank, world).cpu().numpy()))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_two_ranks_learn_the_table_of_one_process():
    import socket
    import torch.multiprocessing as mp
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
    a, b = (torch.from_numpy(r[1]) for r in res)
    assert torch.equal(a, b)                                  # every rank keeps the same table
    single = _dp_cameras(0, 1).cpu()
    for k in range(3):                                        # param, exp_avg, exp_avg_sq; summation order only
        assert _close(a[:, 7 * k:7 * k + 7], single[:, 7 * k:7 * k + 7]), (k, (a - single).abs().max())
