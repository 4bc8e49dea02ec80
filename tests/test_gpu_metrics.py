"""Evaluation image metrics (rdg_image_metrics, rodygs_b200.metrics.image_metrics) and SplatTrainStep.evaluate.

The reference is a float64 twin of the definitions written with F.conv2d / F.avg_pool2d (piqa's conventions as
INTEGRATION.md "Scoring held-out views" states them), pinned to closed forms on the CPU.  On the GPU the kernel meets the
project's value bar against it: 2e-6 relative to float64, or 1.5 x the error of the same twin run in float32."""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

MS_WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)


# ================================================================ twin (device-agnostic) ==

def _taps(dtype, device):
    """The normalised 11-tap Gaussian, sigma 1.5, normalised in float64 and rounded to `dtype`.  (Taps normalised in float32
    sum to 1 only within an ulp; in float64 arithmetic that leaves a variance a^2 S (1 - S) on a flat image, which would
    make the float64 twin's cs differ from 1 by ~1e-5 there.)"""
    g = torch.exp(-((torch.arange(11, dtype=torch.float64) - 5) ** 2) / (2 * 1.5 ** 2))
    return (g / g.sum()).to(dtype=dtype, device=device)


def _ss_cs(x, y, C1, C2):
    """Per-channel means of the SSIM and contrast-structure maps over the valid region: two [B, C] tensors."""
    ch = x.shape[1]
    taps = _taps(x.dtype, x.device)

    def blur(t):
        t = F.conv2d(t, taps.view(1, 1, 1, -1).expand(ch, 1, 1, 11), groups=ch)
        return F.conv2d(t, taps.view(1, 1, -1, 1).expand(ch, 1, 11, 1), groups=ch)

    mx, my = blur(x), blur(y)
    sxx, syy, sxy = blur(x * x) - mx * mx, blur(y * y) - my * my, blur(x * y) - mx * my
    cs = (2 * sxy + C2) / (sxx + syy + C2)
    ss = (2 * mx * my + C1) / (mx * mx + my * my + C1) * cs
    return ss.mean((-1, -2)), cs.mean((-1, -2))


def pyramid(x):
    """The 5 MS-SSIM scales of [B, C, H, W]."""
    out = [x]
    for _ in range(4):
        out.append(F.avg_pool2d(out[-1], 2, ceil_mode=True))
    return out


def twin(pred, gt, value_range=1.0):
    """[B, 4] (mse, psnr, ssim, ms_ssim) in the dtype and on the device of the inputs."""
    x, y = (t if t.dim() == 4 else t[None] for t in (pred, gt))
    R = float(value_range)
    C1, C2 = (0.01 * R) ** 2, (0.03 * R) ** 2
    mse = ((x - y) ** 2).mean((1, 2, 3))
    psnr = 10 * torch.log10(R * R / (mse + 1e-8))
    ss0, _ = _ss_cs(x, y, C1, C2)
    H, W = x.shape[-2:]
    if math.ceil(H / 16) >= 11 and math.ceil(W / 16) >= 11:
        m = torch.ones_like(ss0)
        for s, (xs, ys) in enumerate(zip(pyramid(x), pyramid(y))):
            ss, cs = _ss_cs(xs, ys, C1, C2)
            m = m * (ss if s == 4 else cs).relu() ** MS_WEIGHTS[s]
        ms = m.mean(1)
    else:
        ms = torch.full_like(mse, float("nan"))
    return torch.stack([mse, psnr, ss0.mean(1), ms], 1)


# ================================================================ CPU ==

def test_twin_identical_images():
    x = torch.rand(2, 3, 170, 180, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    out = twin(x, x.clone())
    assert torch.equal(out[:, 0], torch.zeros(2, dtype=torch.float64))
    assert torch.allclose(out[:, 1], torch.full((2,), 80.0, dtype=torch.float64), rtol=0, atol=1e-12)
    assert torch.allclose(out[:, 2:], torch.ones(2, 2, dtype=torch.float64), rtol=0, atol=1e-12)


def test_twin_constant_images_closed_form():
    """Pooling keeps constants, so cs = 1 at every scale and only the last scale's luminance term is left."""
    a, b = 0.3, 0.7
    x, y = torch.full((1, 3, 161, 203), a, dtype=torch.float64), torch.full((1, 3, 161, 203), b, dtype=torch.float64)
    C1 = 0.01 ** 2
    ss = (2 * a * b + C1) / (a * a + b * b + C1)
    for xs, ys in zip(pyramid(x), pyramid(y)):
        _, cs = _ss_cs(xs, ys, C1, 0.03 ** 2)
        assert torch.allclose(cs, torch.ones_like(cs), rtol=0, atol=1e-12)
    out = twin(x, y)[0].tolist()
    assert math.isclose(out[0], (a - b) ** 2, rel_tol=1e-12)
    assert math.isclose(out[1], -10 * math.log10((a - b) ** 2 + 1e-8), rel_tol=1e-12)
    assert math.isclose(out[2], ss, rel_tol=1e-12)
    assert math.isclose(out[3], ss ** 0.1333, rel_tol=1e-12)


@pytest.mark.parametrize("H,W", [(161, 193), (175, 321), (200, 161)])
def test_twin_pyramid_sizes_on_odd_sizes(H, W):
    """ceil(H / 2^s) x ceil(W / 2^s) at every scale, and the window hanging over an odd edge averages its in-bounds pixels
    only (a constant image stays constant)."""
    ones = torch.ones(1, 1, H, W, dtype=torch.float64)
    for s, t in enumerate(pyramid(ones)):
        assert tuple(t.shape[-2:]) == (math.ceil(H / 2 ** s), math.ceil(W / 2 ** s)), s
        assert torch.equal(t, torch.ones_like(t)), s
    assert min(pyramid(ones)[4].shape[-2:]) >= 11


def test_abi_refuses_bad_arguments_without_a_gpu():
    from rodygs_b200 import _lib
    lib = _lib.load()
    one = (C.c_float * 4)()
    ws = lib.rdg_image_metrics_workspace_bytes(2, 3, 161, 193)
    assert ws > 0
    for args, word in (((0, 3, 64, 64), b"batch"), ((1, 0, 64, 64), b"channels"), ((1, 3, 10, 64), b"height"),
                       ((1, 3, 64, 10), b"width")):
        assert lib.rdg_image_metrics_workspace_bytes(*args) == -1
        assert word in lib.rdg_last_error()
        assert lib.rdg_image_metrics(one, one, *args, 1.0, one, one, 1 << 40, None) == -1
        assert word in lib.rdg_last_error()
    good = (2, 3, 161, 193)
    for i, word in ((0, b"pred"), (1, b"gt"), (3, b"out"), (4, b"workspace")):
        ptrs = [one, one, None, one, one]
        ptrs[i] = None
        assert lib.rdg_image_metrics(ptrs[0], ptrs[1], *good, 1.0, ptrs[3], ptrs[4], ws, None) == -1
        assert word in lib.rdg_last_error()
    for vr in (0.0, -1.0, float("nan")):
        assert lib.rdg_image_metrics(one, one, *good, vr, one, one, ws, None) == -1
        assert b"value_range" in lib.rdg_last_error()
    assert lib.rdg_image_metrics(one, one, *good, 1.0, one, one, ws - 1, None) == -1
    assert b"workspace_bytes" in lib.rdg_last_error()
    # below 161 pixels there is no MS-SSIM pyramid to hold, only the scale-0 partial sums
    assert lib.rdg_image_metrics_workspace_bytes(1, 3, 150, 300) < lib.rdg_image_metrics_workspace_bytes(1, 3, 161, 300)


def test_image_metrics_refuses_cpu_tensors():
    from rodygs_b200.metrics import image_metrics
    x = torch.rand(3, 32, 32)
    with pytest.raises(RuntimeError, match="pred is on cpu"):
        image_metrics(x, x)
    if torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="gt is on cpu"):
            image_metrics(x.cuda(), x)


# ================================================================ GPU ==

@pytest.fixture(scope="module")
def no_tf32():
    # the float32 twin sets the allowance where float32 cannot resolve float64: it must not run in TF32
    saved = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32 = saved


def _meets_bar(got, pred, gt, value_range=1.0, nan_ms=False):
    ref64 = twin(pred.double(), gt.double(), value_range).cpu()
    ref32 = twin(pred.float(), gt.float(), value_range).double().cpu()
    got = got.double().cpu()
    cols = 3 if nan_ms else 4
    if nan_ms:
        assert torch.isnan(got[:, 3]).all() and torch.isnan(ref64[:, 3]).all()
    err, err32 = (got[:, :cols] - ref64[:, :cols]).abs(), (ref32[:, :cols] - ref64[:, :cols]).abs()
    bound = torch.maximum(2e-6 * ref64[:, :cols].abs(), 1.5 * err32)
    assert (err <= bound).all(), f"kernel {got[:, :cols].tolist()}\nfloat64 {ref64[:, :cols].tolist()}\nratio {(err / bound).tolist()}"


def _make_step(N, H, W, T=6, seed=3):
    from rodygs_b200 import synthetic
    from rodygs_b200.trainer import SplatTrainStep
    scene = synthetic.to_device(synthetic.make_scene(N, H, W, T, seed=seed), "cuda")
    return SplatTrainStep(scene, H, W, sh_degree=3, w_pearson=0.0)


def _views(step, V, n_views=8):
    from rodygs_b200 import synthetic
    cams = [synthetic.make_camera(v, n_views, step.H, step.W, step.T) for v in range(V)]
    vms = torch.stack([c.world_view_transform.t().contiguous() for c in cams]).cuda()
    pms = torch.stack([c.projection_matrix.t().contiguous() for c in cams]).cuda()
    bts = torch.stack([step.p("table")[c.time_index] for c in cams]).contiguous()
    return cams, vms, pms, bts


def _render(step, cam, vm, pm, bt):
    step.forward_backward(vm, pm, cam.tanfovx, cam.tanfovy, bt, None, None, forward_only=True)
    return step.last_outputs[0].clamp(0.0, 1.0)


@pytest.mark.gpu
def test_kernel_against_twin_1080p_render_and_noise(no_tf32):
    from rodygs_b200.metrics import image_metrics
    H, W = 1080, 1920
    step = _make_step(200_000, H, W)
    cams, vms, pms, bts = _views(step, 1)
    a = _render(step, cams[0], vms[0], pms[0], bts[0]).clone()
    g = torch.Generator(device="cuda").manual_seed(7)
    step.params.add_(torch.randn(step.params.shape, device="cuda", generator=g) * 0.02)    # the perturbed copy
    b = _render(step, cams[0], vms[0], pms[0], bts[0]).clone()
    noise = torch.rand(3, H, W, device="cuda", generator=g)
    pred = torch.stack([a, noise])
    gt = torch.stack([b, 0.5 * noise + 0.5 * torch.rand(3, H, W, device="cuda", generator=g)])
    got = image_metrics(pred, gt)
    _meets_bar(got, pred, gt)
    assert ((got[:, 2] > 0) & (got[:, 2] < 1)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(161, 193), (150, 300)])
def test_kernel_against_twin_odd_and_small_sizes(H, W, no_tf32):
    """161x193: every scale has odd sizes, down to 11x13 (the smallest at which MS-SSIM is defined).  150x300: no MS-SSIM
    (NaN), the other three columns still meet the bar."""
    from rodygs_b200.metrics import image_metrics
    g = torch.Generator(device="cuda").manual_seed(H)
    base = torch.rand(2, 3, H, W, device="cuda", generator=g)
    pred = base
    gt = (base + 0.2 * torch.rand(2, 3, H, W, device="cuda", generator=g)).clamp(0, 1)
    got = image_metrics(pred, gt)
    _meets_bar(got, pred, gt, nan_ms=H < 161)


@pytest.mark.gpu
def test_reproducible_and_independent_of_the_batch():
    from rodygs_b200.metrics import image_metrics
    g = torch.Generator(device="cuda").manual_seed(1)
    pred = torch.rand(3, 3, 200, 333, device="cuda", generator=g)
    gt = torch.rand(3, 3, 200, 333, device="cuda", generator=g) * 0.3 + pred * 0.7
    a, b = image_metrics(pred, gt), image_metrics(pred, gt)
    assert torch.equal(a, b)
    for i in range(3):
        assert torch.equal(image_metrics(pred[i], gt[i])[0], a[i])


@pytest.mark.gpu
def test_value_range(no_tf32):
    from rodygs_b200.metrics import image_metrics
    g = torch.Generator(device="cuda").manual_seed(2)
    pred = torch.rand(2, 3, 170, 190, device="cuda", generator=g)
    gt = (pred + 0.1 * torch.randn(2, 3, 170, 190, device="cuda", generator=g)).clamp(0, 1)
    got = image_metrics(pred * 255, gt * 255, value_range=255)
    ref = twin(pred.double(), gt.double()).cpu()
    ref[:, 0] *= 255 ** 2                        # mse scales with the range squared, psnr / ssim / ms_ssim do not
    got = got.double().cpu()
    _meets_bar(got, pred * 255, gt * 255, value_range=255)
    assert torch.allclose(got, ref, rtol=2e-5, atol=0), (got, ref)


@pytest.mark.gpu
def test_image_metrics_refuses_bad_shapes_and_converts_dtype():
    from rodygs_b200.metrics import image_metrics
    x = torch.rand(3, 40, 40, device="cuda")
    with pytest.raises(ValueError, match="gt has"):
        image_metrics(x, x[:, :39])
    with pytest.raises(ValueError, match="11x11"):
        image_metrics(x[:, :10], x[:, :10])
    with pytest.raises(ValueError, match="pred must be"):
        image_metrics(x[0], x[0])
    # 40x40 is below the MS-SSIM size: that column is NaN in both results, the other three must be the same bits
    a, b = image_metrics(x.double(), x.half().float()), image_metrics(x, x.half().float())
    assert torch.isnan(a[:, 3]).all() and torch.isnan(b[:, 3]).all()
    assert torch.equal(a[:, :3], b[:, :3])


@pytest.mark.gpu
def test_evaluate_rows_are_the_metrics_of_the_clamped_renders():
    from rodygs_b200.metrics import image_metrics
    step = _make_step(20_000, 176, 208)
    cams, vms, pms, bts = _views(step, 3)
    gts = torch.rand(3, 3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4))
    table = step.evaluate(vms, pms, [c.tanfovx for c in cams], cams[0].tanfovy, bts, gts)
    assert table.shape == (3, 4) and table.dtype == torch.float32
    for v, cam in enumerate(cams):
        ref = image_metrics(_render(step, cam, vms[v], pms[v], bts[v]), gts[v])[0]
        assert torch.equal(table[v], ref), (v, table[v], ref)
    assert torch.isfinite(table).all()


def _snapshot(step):
    from rodygs_b200.trainer import STATS_FIELDS
    d = step._deferred
    return {
        "params": step.params.clone(), "grads": step.grads.clone(), "loss_parts": step.loss_parts.clone(),
        "means2D_grad": step.means2D_grad.clone(), "view_grad": step.view_grad.clone(),
        "moments": {t: (o.exp_avg.clone(), o.exp_avg_sq.clone(), o.steps) for t, o in step.optim.items()},
        "stats": {t: [getattr(s, f).clone() for f in STATS_FIELDS] for t, s in step.stats.items()},
        "last_state": step.last_state, "last_outputs": step.last_outputs,
        "outputs": [t.clone() for t in step.last_outputs],
        "rng": torch.cuda.get_rng_state(), "deferred": d, "pending": set(d["pending"]), "dcolor": d["dcolor"].clone(),
        "dc_all": step._dc_all2.clone(), "dcolor_local": step.dcolor_local.clone(),
    }


def _same(a, b):
    if torch.is_tensor(a):
        return torch.equal(a, b)
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(_same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    return a == b


@pytest.mark.gpu
def test_evaluate_leaves_the_training_state_alone():
    """Between forward_backward (+ exchange_grads(defer_sh=True)) and add_densification_stats, with densification and both
    optimisers attached: every piece of training state is bit-identical after evaluate, the objects the next calls read
    (last_state, last_outputs, the deferred factors) are the same objects."""
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
    table = step.evaluate(vms, pms, cams[0].tanfovx, cams[0].tanfovy, bts, gts)
    torch.cuda.synchronize()
    after = _snapshot(step)
    assert torch.isfinite(table).all()
    assert after["last_state"] is before["last_state"] and after["deferred"] is before["deferred"]
    assert all(x is y for x, y in zip(after["last_outputs"], before["last_outputs"]))
    for key in before:
        assert _same(before[key], after[key]), key
    for tag in ("static", "dynamic"):                    # the step carries on as if evaluate had not run
        step.add_densification_stats(tag)
        step.optimizer_step(tag, 2)
    assert not step._deferred["pending"]


@pytest.mark.gpu
def test_evaluate_leaves_a_pending_sync_free_count_and_the_capacity_alone():
    """With config.sync_free the training step leaves its duplicate count unread.  evaluate bins every view at its own
    count: with the capacity cut below any view's count it returns the right rows, leaves the capacity and the pending
    count as they were, and the next training steps (which grow the capacity from that count) do not raise."""
    from rodygs_b200 import engine
    step = _make_step(20_000, 176, 208)
    cams, vms, pms, bts = _views(step, 2)
    g = torch.Generator(device="cuda").manual_seed(6)
    gt = torch.rand(3, 176, 208, device="cuda", generator=g)
    gts = torch.rand(2, 3, 176, 208, device="cuda", generator=g)
    ref = step.evaluate(vms, pms, cams[0].tanfovx, cams[0].tanfovy, bts, gts)
    saved = engine.config.sync_free
    engine.config.sync_free = True
    try:
        for _ in range(2):
            step.forward_backward(vms[0], pms[0], cams[0].tanfovx, cams[0].tanfovy, bts[0], gt, None)
        cap = engine._cap_state(step.params.device, step.ns + step.nd)
        assert cap["pending"] is not None
        pending = cap["pending"]
        cap["cap"] = 256
        table = step.evaluate(vms, pms, cams[0].tanfovx, cams[0].tanfovy, bts, gts)
        assert cap["cap"] == 256 and cap["pending"] is pending
        assert torch.equal(table, ref)
        for _ in range(2):
            lp = step.forward_backward(vms[0], pms[0], cams[0].tanfovx, cams[0].tanfovy, bts[0], gt, None)
        torch.cuda.synchronize()
        assert math.isfinite(float(lp[0]))
    finally:
        engine.config.sync_free = saved
        engine._check_pending(engine._cap_state(step.params.device, step.ns + step.nd))


def _dp_eval_worker(rank, world, port, ret):
    """Two ranks on ONE GPU (gloo carries the CUDA tensors through the host)."""
    import os
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ret.put((rank, _dp_eval_table().cpu().numpy()))
    finally:
        dist.destroy_process_group()


def _dp_eval_table():
    step = _make_step(12_000, 176, 208)
    cams, vms, pms, bts = _views(step, 3)
    gts = torch.rand(3, 3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
    return step.evaluate(vms, pms, [c.tanfovx for c in cams], [c.tanfovy for c in cams], bts, gts)


@pytest.mark.gpu
def test_evaluate_on_two_ranks_matches_one_process():
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    procs = [ctx.Process(target=_dp_eval_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([ret.get(timeout=300), ret.get(timeout=300)], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    single = _dp_eval_table().cpu()
    a, b = (torch.from_numpy(r[1]) for r in res)
    assert torch.equal(a, b), (a, b)
    assert torch.equal(a, single), (a, single)
