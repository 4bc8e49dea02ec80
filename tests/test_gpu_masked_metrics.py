"""Masked evaluation metrics over a covisibility mask (rdg_masked_image_metrics, rodygs_b200.metrics.masked_image_metrics)
and SplatTrainStep.evaluate(masks=).

The reference is a float64 twin of DyCheck's masked PSNR / SSIM as INTEGRATION.md "Scoring held-out views" states them,
written with F.conv2d (a ones kernel for the counts) and pinned to closed forms on the CPU.  On the GPU the kernel meets the
project's value bar against it: 2e-6 relative to float64, or 1.5 x the error of the same twin run in float32."""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

from test_gpu_metrics import _make_step, _render, _same, _snapshot, _views
from test_gpu_metrics import twin as piqa_twin


# ================================================================ twin (device-agnostic) ==

def _taps(dtype, device):
    g = torch.exp(-((torch.arange(11, dtype=torch.float64) - 5) ** 2) / (2 * 1.5 ** 2))
    return (g / g.sum()).to(dtype=dtype, device=device)


def partial_blur(z, m):
    """P(z): the two-stage valid partial convolution.  z [N, H, W], m [N, H, W] -> [N, H - 10, W - 10]."""
    z, m = z[:, None], m[:, None]
    g = _taps(z.dtype, z.device)
    ones = torch.ones(11, dtype=z.dtype, device=z.device)
    zero = torch.zeros((), dtype=z.dtype, device=z.device)
    n1 = F.conv2d(m, ones.view(1, 1, 1, 11))
    p1 = torch.where(n1 != 0, F.conv2d(m * z, g.view(1, 1, 1, 11)) * 11 / n1, zero)
    v1 = (n1 != 0).to(z.dtype)
    n2 = F.conv2d(v1, ones.view(1, 1, 11, 1))
    return torch.where(n2 != 0, F.conv2d(v1 * p1, g.view(1, 1, 11, 1)) * 11 / n2, zero)[:, 0]


def twin(pred, gt, mask, value_range=1.0):
    """[B, 3] (mmse, mpsnr, mssim) in the dtype and on the device of the inputs; mask [B, 1, H, W] or [1, H, W]."""
    x, y, m = (t if t.dim() == 4 else t[None] for t in (pred, gt, mask))
    m = m.to(x.dtype)
    B, Cc, H, W = x.shape
    R = float(value_range)
    C1, C2 = (0.01 * R) ** 2, (0.03 * R) ** 2
    mb = m.expand(B, Cc, H, W)
    keep = mb != 0
    x, y = torch.where(keep, x, 0.0), torch.where(keep, y, 0.0)        # masked-out values take no part, NaN included
    mmse = (mb * (x - y) ** 2).sum((1, 2, 3)) / (Cc * m.sum((1, 2, 3)))
    flat = [t.reshape(B * Cc, H, W) for t in (x, y, mb)]
    P = lambda z: partial_blur(z, flat[2]).view(B, Cc, H - 10, W - 10)   # noqa: E731
    xf, yf = flat[0], flat[1]
    mx, my = P(xf), P(yf)
    sxx, syy = (P(xf * xf) - mx * mx).clamp(min=0), (P(yf * yf) - my * my).clamp(min=0)
    s = P(xf * yf) - mx * my
    sxy = torch.sign(s) * torch.minimum((sxx * syy).sqrt(), s.abs())
    ssim_map = (2 * mx * my + C1) * (2 * sxy + C2) / ((mx * mx + my * my + C1) * (sxx + syy + C2))
    return torch.stack([mmse, 10 * torch.log10(R * R / mmse), ssim_map.mean((1, 2, 3))], 1)


def covisibility_mask(B, H, W, gen, device):
    """Blobs with ragged edges and single-pixel holes, about half the image covisible."""
    low = torch.rand(B, 1, H // 40 + 2, W // 40 + 2, device=device, generator=gen)
    smooth = F.interpolate(low, size=(H, W), mode="bilinear", align_corners=False)
    ragged = smooth + 0.1 * torch.rand(B, 1, H, W, device=device, generator=gen)
    holes = torch.rand(B, 1, H, W, device=device, generator=gen) < 0.01
    return ((ragged > 0.55) & ~holes).float()


# ================================================================ CPU ==

def _pair64(B, H, W, seed):
    gen = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 3, H, W, dtype=torch.float64, generator=gen)
    y = (x + 0.2 * torch.rand(B, 3, H, W, dtype=torch.float64, generator=gen)).clamp(0, 1)
    return x, y, gen


def test_twin_all_ones_mask_is_the_unmasked_ssim_and_mse():
    x, y, _ = _pair64(2, 64, 80, 0)
    got = twin(x, y, torch.ones(2, 1, 64, 80, dtype=torch.float64))
    ref = piqa_twin(x, y)
    assert torch.allclose(got[:, 2], ref[:, 2], rtol=0, atol=1e-12)
    assert torch.allclose(got[:, 0], ref[:, 0], rtol=1e-12, atol=0)


def test_twin_empty_mask():
    x, y, _ = _pair64(2, 40, 50, 1)
    got = twin(x, y, torch.zeros(2, 1, 40, 50, dtype=torch.float64))
    assert torch.isnan(got[:, :2]).all()
    assert torch.equal(got[:, 2], torch.ones(2, dtype=torch.float64))


def test_twin_partial_blur_of_one_at_a_lone_pixel():
    """P(1) is not 1: at the window centred on a lone covisible pixel it is 121 g_5^2 (about 8.56), and 121 g_s g_t at the
    window that holds it at tap (s, t)."""
    g = _taps(torch.float64, "cpu")
    m = torch.zeros(1, 41, 41, dtype=torch.float64)
    m[0, 20, 20] = 1
    p = partial_blur(torch.ones_like(m), m)[0]
    assert math.isclose(p.max().item(), 121 * g[5].item() ** 2, rel_tol=1e-12)
    expect = torch.zeros(31, 31, dtype=torch.float64)
    expect[10:21, 10:21] = 121 * torch.outer(g, g).flip(0, 1)
    assert torch.allclose(p, expect, rtol=1e-12, atol=0)


def test_twin_constant_images_under_a_one_pixel_mask_closed_form():
    a, b = 0.3, 0.7
    x, y = torch.full((1, 3, 41, 41), a, dtype=torch.float64), torch.full((1, 3, 41, 41), b, dtype=torch.float64)
    m = torch.zeros(1, 1, 41, 41, dtype=torch.float64)
    m[0, 0, 20, 20] = 1
    g = _taps(torch.float64, "cpu").tolist()
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    total = 31 * 31 - 121                                 # windows without the pixel score exactly 1
    for s in range(11):
        for t in range(11):
            q = 121 * g[s] * g[t]                         # P(1) of that window
            var = max(0.0, q * (1 - q))                   # clipped where P(1) > 1
            num = (2 * a * b * q * q + C1) * (2 * a * b * var + C2)
            total += num / (((a * a + b * b) * q * q + C1) * ((a * a + b * b) * var + C2))
    out = twin(x, y, m)[0].tolist()
    assert math.isclose(out[0], (a - b) ** 2, rel_tol=1e-12)
    assert math.isclose(out[1], -10 * math.log10((a - b) ** 2), rel_tol=1e-12)
    assert math.isclose(out[2], total / (31 * 31), rel_tol=1e-12)


def test_twin_ignores_masked_out_values_and_clipping_matters():
    x, y, gen = _pair64(2, 64, 80, 2)
    m = (torch.rand(2, 1, 64, 80, dtype=torch.float64, generator=gen) > 0.4).double()
    ref = twin(x, y, m)
    out = m.expand_as(x) == 0
    x2 = torch.where(out, torch.rand(x.shape, dtype=torch.float64, generator=gen), x)
    y2 = torch.where(out, torch.full_like(y, float("nan")), y)
    assert torch.equal(twin(x2, y2, m), ref)
    # a random 60 % mask leaves a negative raw variance at a few percent of the positions
    raw = partial_blur((x * x)[:, 0], m[:, 0]) - partial_blur(x[:, 0], m[:, 0]) ** 2
    assert 0.005 < (raw < 0).double().mean().item() < 0.1


def test_abi_refuses_bad_arguments_without_a_gpu():
    from rodygs_b200 import _lib
    lib = _lib.load()
    one = (C.c_float * 4)()
    ws = lib.rdg_masked_image_metrics_workspace_bytes(2, 3, 161, 193)
    assert ws > 0
    for args, word in (((0, 3, 64, 64), b"batch"), ((1, 0, 64, 64), b"channels"), ((1, 3, 10, 64), b"height"),
                       ((1, 3, 64, 10), b"width")):
        assert lib.rdg_masked_image_metrics_workspace_bytes(*args) == -1
        assert word in lib.rdg_last_error()
        assert lib.rdg_masked_image_metrics(one, one, one, *args, 1.0, one, one, 1 << 40, None) == -1
        assert word in lib.rdg_last_error()
    good = (2, 3, 161, 193)
    for i, word in ((0, b"pred"), (1, b"gt"), (2, b"mask"), (3, b"out"), (4, b"workspace")):
        ptrs = [one] * 5
        ptrs[i] = None
        assert lib.rdg_masked_image_metrics(ptrs[0], ptrs[1], ptrs[2], *good, 1.0, ptrs[3], ptrs[4], ws, None) == -1
        assert word in lib.rdg_last_error()
    for vr in (0.0, -1.0, float("nan")):
        assert lib.rdg_masked_image_metrics(one, one, one, *good, vr, one, one, ws, None) == -1
        assert b"value_range" in lib.rdg_last_error()
    assert lib.rdg_masked_image_metrics(one, one, one, *good, 1.0, one, one, ws - 1, None) == -1
    assert b"workspace_bytes" in lib.rdg_last_error()


def test_masked_image_metrics_refuses_cpu_tensors():
    from rodygs_b200.metrics import masked_image_metrics
    x, m = torch.rand(3, 32, 32), torch.ones(1, 32, 32)
    with pytest.raises(RuntimeError, match="pred is on cpu"):
        masked_image_metrics(x, x, m)
    if torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="mask is on cpu"):
            masked_image_metrics(x.cuda(), x.cuda(), m)


# ================================================================ GPU ==

@pytest.fixture(scope="module")
def no_tf32():
    # the float32 twin sets the allowance where float32 cannot resolve float64: it must not run in TF32
    saved = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32 = saved


def _meets_bar(got, pred, gt, mask, value_range=1.0):
    ref64 = twin(pred.double(), gt.double(), mask.double(), value_range).cpu()
    ref32 = twin(pred.float(), gt.float(), mask.float(), value_range).double().cpu()
    got = got.double().cpu()
    err, err32 = (got - ref64).abs(), (ref32 - ref64).abs()
    bound = torch.maximum(2e-6 * ref64.abs(), 1.5 * err32)
    assert (err <= bound).all(), f"kernel {got.tolist()}\nfloat64 {ref64.tolist()}\nratio {(err / bound).tolist()}"


def _noise_pair(B, H, W, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    pred = torch.rand(B, 3, H, W, device="cuda", generator=g)
    gt = (pred + 0.2 * torch.rand(B, 3, H, W, device="cuda", generator=g)).clamp(0, 1)
    mask = (torch.rand(B, 1, H, W, device="cuda", generator=g) > 0.4).float()
    return pred, gt, mask, g


@pytest.mark.gpu
def test_kernel_against_twin_1080p_render_and_noise(no_tf32):
    from rodygs_b200.metrics import masked_image_metrics
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
    mask = torch.cat([covisibility_mask(1, H, W, g, "cuda"), (torch.rand(1, 1, H, W, device="cuda", generator=g) > 0.4).float()])
    got = masked_image_metrics(pred, gt, mask)
    _meets_bar(got, pred, gt, mask)
    assert ((got[:, 2] > 0) & (got[:, 2] < 1)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(11, 11), (13, 200), (161, 193), (150, 300)])
def test_kernel_against_twin_small_and_odd_sizes(H, W, no_tf32):
    from rodygs_b200.metrics import masked_image_metrics
    pred, gt, mask, _ = _noise_pair(2, H, W, H * 1000 + W)
    _meets_bar(masked_image_metrics(pred, gt, mask), pred, gt, mask)


@pytest.mark.gpu
def test_kernel_against_twin_fractional_mask(no_tf32):
    from rodygs_b200.metrics import masked_image_metrics
    pred, gt, mask, g = _noise_pair(2, 170, 190, 3)
    mask = mask * torch.rand(mask.shape, device="cuda", generator=g)
    _meets_bar(masked_image_metrics(pred, gt, mask), pred, gt, mask)


@pytest.mark.gpu
def test_value_range(no_tf32):
    from rodygs_b200.metrics import masked_image_metrics
    pred, gt, mask, _ = _noise_pair(2, 170, 190, 4)
    got = masked_image_metrics(pred * 255, gt * 255, mask, value_range=255)
    _meets_bar(got, pred * 255, gt * 255, mask, value_range=255)
    ref = twin(pred.double(), gt.double(), mask.double()).cpu()
    ref[:, 0] *= 255 ** 2                        # mmse scales with the range squared, mpsnr / mssim do not
    assert torch.allclose(got.double().cpu(), ref, rtol=2e-5, atol=0), (got, ref)


@pytest.mark.gpu
def test_all_ones_mask_is_image_metrics():
    from rodygs_b200.metrics import image_metrics, masked_image_metrics
    pred, gt, _, _ = _noise_pair(2, 200, 333, 5)
    got = masked_image_metrics(pred, gt, torch.ones(2, 1, 200, 333, device="cuda")).double().cpu()
    ref = image_metrics(pred, gt).double().cpu()
    for k, j in ((0, 0), (2, 2)):                # mmse = mse, mssim = ssim
        assert torch.allclose(got[:, k], ref[:, j], rtol=2e-6, atol=0), (k, got[:, k], ref[:, j])


@pytest.mark.gpu
def test_empty_mask():
    from rodygs_b200.metrics import masked_image_metrics
    pred, gt, mask, _ = _noise_pair(2, 64, 90, 6)
    got = masked_image_metrics(pred, gt, torch.zeros_like(mask)).cpu()
    assert torch.isnan(got[:, :2]).all()
    assert torch.equal(got[:, 2], torch.ones(2))


@pytest.mark.gpu
def test_masked_out_values_change_no_bit():
    from rodygs_b200.metrics import masked_image_metrics
    pred, gt, mask, g = _noise_pair(2, 150, 170, 7)
    ref = masked_image_metrics(pred, gt, mask)
    out = mask.expand_as(pred) == 0
    for fill in (torch.rand(pred.shape, device="cuda", generator=g) * 100 - 50,
                 torch.full_like(pred, float("nan")), torch.full_like(pred, float("inf")),
                 torch.full_like(pred, -float("inf"))):
        got = masked_image_metrics(torch.where(out, fill, pred), torch.where(out, fill.flip(-1), gt), mask)
        assert torch.equal(got, ref), (got, ref)


@pytest.mark.gpu
def test_reproducible_and_independent_of_the_batch():
    from rodygs_b200.metrics import masked_image_metrics
    pred, gt, mask, _ = _noise_pair(3, 200, 333, 8)
    a, b = masked_image_metrics(pred, gt, mask), masked_image_metrics(pred, gt, mask)
    assert torch.equal(a, b)
    for i in range(3):
        assert torch.equal(masked_image_metrics(pred[i], gt[i], mask[i])[0], a[i])


@pytest.mark.gpu
def test_mask_dtypes_and_shapes():
    from rodygs_b200.metrics import masked_image_metrics
    pred, gt, mask, _ = _noise_pair(2, 60, 70, 9)
    ref = masked_image_metrics(pred, gt, mask)
    for m in (mask.bool(), mask.to(torch.uint8), mask.double(), mask.half()):
        assert torch.equal(masked_image_metrics(pred, gt, m), ref), m.dtype
    with pytest.raises(ValueError, match="mask must have shape"):
        masked_image_metrics(pred, gt, mask[:, 0])
    with pytest.raises(ValueError, match="mask must have shape"):
        masked_image_metrics(pred, gt, mask.expand(2, 3, 60, 70))
    with pytest.raises(ValueError, match="mask must have shape"):
        masked_image_metrics(pred[0], gt[0], mask)
    with pytest.raises(ValueError, match="gt has"):
        masked_image_metrics(pred, gt[..., :69], mask)


def _masks(V, H, W, seed):
    return covisibility_mask(V, H, W, torch.Generator(device="cuda").manual_seed(seed), "cuda")


@pytest.mark.gpu
def test_evaluate_with_masks_adds_the_masked_columns():
    from rodygs_b200.metrics import masked_image_metrics
    step = _make_step(20_000, 176, 208)
    cams, vms, pms, bts = _views(step, 3)
    gts = torch.rand(3, 3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4))
    masks = _masks(3, 176, 208, 5)
    fx = [c.tanfovx for c in cams]
    plain = step.evaluate(vms, pms, fx, cams[0].tanfovy, bts, gts)
    table = step.evaluate(vms, pms, fx, cams[0].tanfovy, bts, gts, masks=masks)
    assert table.shape == (3, 7) and table.dtype == torch.float32
    assert torch.equal(table[:, :4], plain)
    for v, cam in enumerate(cams):
        ref = masked_image_metrics(_render(step, cam, vms[v], pms[v], bts[v]), gts[v], masks[v])[0]
        assert torch.equal(table[v, 4:], ref), (v, table[v], ref)
    assert torch.isfinite(table).all()
    with pytest.raises(ValueError, match="masks must be"):
        step.evaluate(vms, pms, fx, cams[0].tanfovy, bts, gts, masks=masks[:2])


@pytest.mark.gpu
def test_evaluate_with_masks_leaves_the_training_state_alone():
    """As test_gpu_metrics.test_evaluate_leaves_the_training_state_alone, with masks."""
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
    table = step.evaluate(vms, pms, cams[0].tanfovx, cams[0].tanfovy, bts, gts, masks=_masks(3, 176, 208, 6))
    torch.cuda.synchronize()
    after = _snapshot(step)
    assert table.shape == (3, 7) and torch.isfinite(table).all()
    assert after["last_state"] is before["last_state"] and after["deferred"] is before["deferred"]
    assert all(x is y for x, y in zip(after["last_outputs"], before["last_outputs"]))
    for key in before:
        assert _same(before[key], after[key]), key
    for tag in ("static", "dynamic"):
        step.add_densification_stats(tag)
        step.optimizer_step(tag, 2)
    assert not step._deferred["pending"]


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
    return step.evaluate(vms, pms, [c.tanfovx for c in cams], [c.tanfovy for c in cams], bts, gts,
                         masks=_masks(3, 176, 208, 9))


@pytest.mark.gpu
def test_evaluate_with_masks_on_two_ranks_matches_one_process():
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
    assert a.shape == (3, 7)
    assert torch.equal(a, b), (a, b)
    assert torch.equal(a, single), (a, single)
