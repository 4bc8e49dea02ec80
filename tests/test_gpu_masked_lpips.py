"""Masked LPIPS over a covisibility mask, DyCheck's mLPIPS (rdg_masked_lpips, rodygs_b200.metrics.masked_lpips) and
SplatTrainStep.evaluate(masked_lpips=).

The reference is a float64 twin of the definition INTEGRATION.md "Scoring held-out views" states: the LPIPS twin of
test_gpu_lpips on masked inputs, each tap's head map upsampled with F.interpolate(mode="bilinear", align_corners=False),
summed, and averaged under the mask.  It is pinned to closed forms on the CPU.  On the GPU the kernel must agree with the
twin that rounds each conv's operands to TF32 as the kernel does to 1e-4 relative, and with the plain float64 twin (the cost
of TF32) to 5e-3, as rdg_lpips does."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from test_gpu_lpips import GEOM, POOLS, TAPS, _render_pair, random_weights, rna_tf32, twin
from test_gpu_masked_metrics import covisibility_mask
from test_gpu_metrics import _make_step, _render, _same, _snapshot, _views

from rodygs_b200.metrics import LPIPS_CONVS


# ================================================================ twin ==

def head_maps(pred, gt, bb, lin, net, value_range=1.0, tf32=False):
    """The lpips head at every position of each tap, [B, h_l, w_l] float64 per tap; pred, gt [B, 3, H, W].  The same
    network as test_gpu_lpips.twin, which is the mean of each map summed over the taps."""
    dev = pred.device
    mu = torch.tensor([0.485, 0.456, 0.406], dtype=torch.float64, device=dev).view(1, 3, 1, 1)
    sd = torch.tensor([0.229, 0.224, 0.225], dtype=torch.float64, device=dev).view(1, 3, 1, 1)
    z = (torch.cat([pred, gt]).double() / value_range - mu) / sd
    B = pred.shape[0]
    maps = []
    for i, _, _, _ in LPIPS_CONVS[net]:
        if i in POOLS[net]:
            z = F.max_pool2d(z, POOLS[net][i], 2)
        w = bb[f"features.{i}.weight"].to(dev, torch.float64)
        b = bb[f"features.{i}.bias"].to(dev, torch.float64)
        s, p = GEOM.get(net, {}).get(i, (1, 1))
        z = F.relu(F.conv2d(rna_tf32(z) if tf32 else z, rna_tf32(w) if tf32 else w, b, stride=s, padding=p))
        if i in TAPS[net]:
            n = z / (z.pow(2).sum(1, keepdim=True).sqrt() + 1e-10)
            wl = lin[f"lin{len(maps)}.model.1.weight"].to(dev, torch.float64)
            maps.append((wl * (n[:B] - n[B:]) ** 2).sum(1))
    return maps


def masked_twin(pred, gt, mask, bb, lin, net, value_range=1.0, tf32=False):
    """[B] masked LPIPS in float64 on the device of the inputs; pred, gt [B, 3, H, W], mask [B, 1, H, W]."""
    m = mask.double()
    keep = m != 0
    x, y = (torch.where(keep, m * t.double(), 0.0) for t in (pred, gt))    # masked-out values take no part, NaN included
    H, W = pred.shape[-2:]
    spatial = sum(F.interpolate(d[:, None], size=(H, W), mode="bilinear", align_corners=False)
                  for d in head_maps(x, y, bb, lin, net, value_range, tf32))
    return (m * spatial).sum((1, 2, 3)) / m.sum((1, 2, 3))


def _pair64(B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 3, H, W, dtype=torch.float64, generator=g)
    y = (x + 0.2 * torch.randn(B, 3, H, W, dtype=torch.float64, generator=g)).clamp(0, 1)
    m = covisibility_mask(B, H, W, g, "cpu").double()
    return x, y, m, g


# ================================================================ CPU ==

@pytest.mark.parametrize("n_in,n_out", [(15, 64), (7, 97), (64, 64), (32, 64), (269, 1080), (33, 131)])
def test_interpolate_is_the_stated_bilinear_formula(n_in, n_out):
    """F.interpolate(bilinear, align_corners=False) per axis: src = max(scale (dst + 0.5) - 0.5, 0), i0 = floor(src),
    i1 = min(i0 + 1, in - 1), weights (1 - l1, l1) with l1 = src - i0, scale = in / out; the 2-D result is the product."""
    A = torch.zeros(n_out, n_in, dtype=torch.float64)
    scale = n_in / n_out
    for dst in range(n_out):
        src = max(scale * (dst + 0.5) - 0.5, 0.0)
        i0 = int(src)
        i1 = min(i0 + 1, n_in - 1)
        l1 = src - i0
        A[dst, i0] += 1 - l1
        A[dst, i1] += l1
    g = torch.Generator().manual_seed(n_in * 1000 + n_out)
    d = torch.rand(2, n_in, n_in + 3, dtype=torch.float64, generator=g)
    B = torch.zeros(n_out + 5, n_in + 3, dtype=torch.float64)
    s = (n_in + 3) / (n_out + 5)
    for dst in range(n_out + 5):
        src = max(s * (dst + 0.5) - 0.5, 0.0)
        i0 = int(src)
        l1 = src - i0
        B[dst, i0] += 1 - l1
        B[dst, min(i0 + 1, n_in + 2)] += l1
    got = F.interpolate(d[:, None], size=(n_out, n_out + 5), mode="bilinear", align_corners=False)[:, 0]
    assert torch.allclose(got, A @ d @ B.T, rtol=0, atol=1e-12)


def test_head_maps_are_the_lpips_twin_per_position():
    for net in ("alex", "vgg"):
        bb, lin = random_weights(net, 30)
        x, y, _, _ = _pair64(2, 64, 72, 1)
        maps = head_maps(x, y, bb, lin, net)
        assert [tuple(d.shape[1:]) for d in maps][0] == ((15, 17) if net == "alex" else (64, 72))
        assert torch.allclose(sum(d.mean((1, 2)) for d in maps), twin(x, y, bb, lin, net), rtol=1e-12, atol=0)


def test_twin_closed_forms():
    for net in ("alex", "vgg"):
        bb, lin = random_weights(net, 31)
        x, y, m, g = _pair64(2, 64, 64, 2)
        ref = masked_twin(x, y, m, bb, lin, net)
        assert (ref > 0).all() and torch.isfinite(ref).all()
        assert torch.equal(masked_twin(x, x, m, bb, lin, net), torch.zeros(2, dtype=torch.float64))
        assert torch.isnan(masked_twin(x, y, torch.zeros_like(m), bb, lin, net)).all()
        out = m.expand_as(x) == 0
        x2 = torch.where(out, torch.rand(x.shape, dtype=torch.float64, generator=g), x)
        y2 = torch.where(out, torch.full_like(y, float("nan")), y)
        assert torch.equal(masked_twin(x2, y2, m, bb, lin, net), ref)
        # the images differ in the last 6 columns only, where the clamped upsampling weighs the maps unevenly
        y_edge = torch.cat([x[..., :-6], y[..., -6:]], -1)
        ones = masked_twin(x, y_edge, torch.ones_like(m), bb, lin, net)
        plain = twin(x, y_edge, bb, lin, net)
        rel = ((ones - plain).abs() / plain).min().item()
        if net == "vgg":
            # taps 64, 32, 16, 8, 4 all divide 64: bilinear upsampling with align_corners=False keeps each map's mean
            assert ((ones - plain).abs() / plain).max().item() <= 1e-12
        else:
            # alex's taps at 64x64 are 15, 7, 3, 3, 3: upsampled, not pooled, so the mean moves
            assert rel > 3e-4, rel


def test_masked_lpips_refuses_cpu_tensors_mask_shapes_channels_and_small_sizes():
    from rodygs_b200.metrics import LpipsWeights, masked_lpips
    for net, edge in (("alex", 31), ("vgg", 16)):
        w = LpipsWeights(net, torch.zeros(1))
        x, m = torch.rand(3, 40, 40), torch.ones(1, 40, 40)
        with pytest.raises(RuntimeError, match="pred is on cpu"):
            masked_lpips(x, x, m, w)
        with pytest.raises(ValueError, match="mask must have shape"):
            masked_lpips(x, x, m[0], w)
        with pytest.raises(ValueError, match="mask must have shape"):
            masked_lpips(x[None].expand(2, 3, 40, 40), x[None].expand(2, 3, 40, 40), m, w)
        with pytest.raises(ValueError, match="3 channels"):
            masked_lpips(torch.rand(2, 4, 40, 40), torch.rand(2, 4, 40, 40), torch.ones(2, 1, 40, 40), w)
        with pytest.raises(ValueError, match=f">= {edge}"):
            masked_lpips(torch.rand(3, edge - 1, 64), torch.rand(3, edge - 1, 64), torch.ones(1, edge - 1, 64), w)
        with pytest.raises(ValueError, match=f">= {edge}"):
            masked_lpips(torch.rand(1, 3, 64, edge - 1), torch.rand(1, 3, 64, edge - 1), torch.ones(1, 1, 64, edge - 1), w)
    with pytest.raises(TypeError, match="LpipsWeights"):
        masked_lpips(torch.rand(3, 40, 40), torch.rand(3, 40, 40), torch.ones(1, 40, 40), None)
    with pytest.raises(TypeError, match="mask must be a tensor"):
        masked_lpips(torch.rand(3, 40, 40), torch.rand(3, 40, 40), None, LpipsWeights("alex", torch.zeros(1)))


def test_abi_refuses_bad_arguments_without_a_gpu():
    from rodygs_b200 import _lib
    lib = _lib.load()
    one = (C.c_float * 4)()
    alex, vgg = 0, 1
    n_alex, n_vgg = lib.rdg_lpips_packed_floats(alex), lib.rdg_lpips_packed_floats(vgg)
    assert lib.rdg_masked_lpips_workspace_bytes(alex, 31, 31) > 0 and lib.rdg_masked_lpips_workspace_bytes(vgg, 16, 16) > 0
    for args, word in (((2, 64, 64), b"net"), ((alex, 30, 64), b"height"), ((alex, 64, 30), b"width"),
                       ((vgg, 15, 64), b"height"), ((vgg, 64, 15), b"width"), ((vgg, 1 << 14, 1 << 13), b"2^26")):
        assert lib.rdg_masked_lpips_workspace_bytes(*args) == -1
        assert word in lib.rdg_last_error() and b"rdg_masked_lpips_workspace_bytes" in lib.rdg_last_error()
    ws = lib.rdg_masked_lpips_workspace_bytes(vgg, 64, 80)

    def call(pred=one, gt=one, mask=one, B=2, Cc=3, H=64, W=80, vr=1.0, net=vgg, packed=one, nf=n_vgg, out=one, w=one, nb=ws):
        return lib.rdg_masked_lpips(pred, gt, mask, B, Cc, H, W, vr, net, packed, nf, out, w, nb, None)

    for kw, word in ((dict(pred=None), b"pred"), (dict(gt=None), b"gt"), (dict(mask=None), b"mask"),
                     (dict(packed=None), b"packed"), (dict(out=None), b"out"), (dict(w=None), b"workspace"),
                     (dict(net=5), b"net"), (dict(B=0), b"batch"), (dict(Cc=1), b"channels"), (dict(Cc=4), b"channels"),
                     (dict(H=15), b"height"), (dict(W=15), b"width"), (dict(vr=0.0), b"value_range"),
                     (dict(vr=float("inf")), b"value_range"), (dict(vr=float("nan")), b"value_range"),
                     (dict(nf=n_vgg - 1), b"packed_floats"), (dict(nf=n_alex), b"packed_floats"),
                     (dict(nb=ws - 1), b"rdg_masked_lpips_workspace_bytes()")):
        assert call(**kw) == -1, kw
        err = lib.rdg_last_error()
        assert word in err and err.startswith(b"rdg_masked_lpips:"), (kw, err)
    # rdg_lpips' workspace is not enough for the masked call at a size where the maps outgrow the head slots
    small = lib.rdg_lpips_workspace_bytes(alex, 1080, 1920)
    big = lib.rdg_masked_lpips_workspace_bytes(alex, 1080, 1920)
    assert big > small
    assert call(net=alex, H=1080, W=1920, nf=n_alex, nb=small) == -1 and b"workspace_bytes" in lib.rdg_last_error()


def test_workspace_sizes_above_2_gib_without_a_gpu():
    """Workspaces past 2^31 bytes come back whole: vgg needs about 1 KB per pixel, so 1440x2560 is already past it.  The
    plain sizes are rdg_lpips_workspace_bytes' values before the masked path was added."""
    from rodygs_b200 import _lib
    lib = _lib.load()
    alex, vgg = 0, 1
    for net, H, W, plain in ((vgg, 1440, 2560, 3774920960), (vgg, 2160, 3840, 8493512960), (alex, 8000, 8000, 4091952384)):
        assert lib.rdg_lpips_workspace_bytes(net, H, W) == plain, (net, H, W)
        masked = lib.rdg_masked_lpips_workspace_bytes(net, H, W)
        assert masked >= plain > 1 << 31, (net, H, W, masked)


def test_masked_kernels_do_not_spill():
    """`-Xptxas -v` for the kernels the masked path adds or changes: no spills, no stack frame."""
    import os
    import re
    import subprocess
    import tempfile
    from rodygs_b200 import build
    with tempfile.TemporaryDirectory() as tmp:
        r = subprocess.run([build._nvcc(), *build.ARCH, *build.COMMON, "-Xptxas", "-v", "-c",
                            os.path.join(build.CSRC, "lpips.cu"), "-o", os.path.join(tmp, "lpips.o")],
                           capture_output=True, text=True, check=True)
    info = {}
    name = None
    for line in r.stderr.splitlines():
        hit = re.search(r"Compiling entry function '(\w+)'", line)
        if hit:
            name = hit.group(1)
        elif name and "spill" in line:
            info[name] = line.strip()
    new = [n for n in info if any(k in n for k in ("lpips_spatial_kernel", "lpips_masked_finalize_kernel",
                                                   "lpips_head_kernelILb1", "lpips_scale_kernel"))]
    assert len(new) == 4, sorted(info)
    for n in new:
        assert info[n] == "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads", (n, info[n])


# ================================================================ GPU ==

@pytest.fixture(scope="module")
def no_tf32():
    saved = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32 = saved


@pytest.fixture(scope="module")
def nets():
    from rodygs_b200.metrics import load_lpips
    out = {}
    for k, net in enumerate(("alex", "vgg")):
        bb, lin = random_weights(net, 40 + k)
        out[net] = (load_lpips(net, bb, lin), bb, lin)
    return out


def _masked_pair(H, W, seed):
    pred, gt = _render_pair(H, W, 20_000 if H < 200 else 150_000, seed)
    mask = covisibility_mask(1, H, W, torch.Generator(device="cuda").manual_seed(seed + 1), "cuda")
    return pred, gt, mask


@pytest.mark.gpu
@pytest.mark.parametrize("net,H,W", [("alex", 64, 64), ("vgg", 64, 64), ("alex", 97, 131), ("vgg", 97, 131),
                                     ("alex", 1080, 1920), ("vgg", 540, 960)])
def test_kernel_against_the_twin(net, H, W, nets, no_tf32):
    """1e-4 relative against the twin with the kernel's TF32 operand rounding; 5e-3 against the plain float64 twin."""
    from rodygs_b200.metrics import masked_lpips
    w, bb, lin = nets[net]
    pred, gt, mask = _masked_pair(H, W, H + W)
    cover = mask.mean().item()
    assert 0.2 < cover < 0.8, cover
    got = masked_lpips(pred, gt, mask, w).double()
    ref_tf32 = masked_twin(pred, gt, mask, bb, lin, net, tf32=True)
    ref64 = masked_twin(pred, gt, mask, bb, lin, net)
    layout = ((got - ref_tf32).abs() / ref_tf32.abs()).max().item()
    cost = ((got - ref64).abs() / ref64.abs()).max().item()
    print(f"\n{net} {H}x{W} ({cover:.2f} covisible): kernel {got.tolist()} tf32-twin {ref_tf32.tolist()} "
          f"float64 {ref64.tolist()} rel err vs tf32 twin {layout:.3e}, vs float64 {cost:.3e}")
    assert got.item() > 0
    assert layout <= 1e-4, (net, H, W, layout)
    assert cost <= 5e-3, (net, H, W, cost)


@pytest.mark.gpu
def test_exact_properties(nets):
    from rodygs_b200.metrics import masked_lpips
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.rand(3, 3, 70, 90, device="cuda", generator=g)
    y = (x + 0.1 * torch.randn(x.shape, device="cuda", generator=g)).clamp(0, 1)
    m = covisibility_mask(3, 70, 90, g, "cuda")
    out = m.expand_as(x) == 0
    for net in ("alex", "vgg"):
        w = nets[net][0]
        assert torch.equal(masked_lpips(x, x, m, w), torch.zeros(3, device="cuda"))
        a, b = masked_lpips(x, y, m, w), masked_lpips(x, y, m, w)
        assert torch.equal(a, b)
        assert a.shape == (3,) and a.dtype == torch.float32 and (a > 0).all()
        for i in range(3):
            assert torch.equal(masked_lpips(x[i], y[i], m[i], w), a[i:i + 1])
        assert torch.isnan(masked_lpips(x, y, torch.zeros_like(m), w)).all()
        for fill in (torch.full_like(x, float("nan")), torch.full_like(x, float("inf")),
                     torch.rand(x.shape, device="cuda", generator=g) * 100 - 50):
            got = masked_lpips(torch.where(out, fill, x), torch.where(out, fill.flip(-1), y), m, w)
            assert torch.equal(got, a), (net, got, a)
        for mm in (m.bool(), m.to(torch.uint8), m.half(), m.double()):
            assert torch.equal(masked_lpips(x, y, mm, w), a), mm.dtype
        r = masked_lpips(255 * x, 255 * y, m, w, value_range=255)
        assert torch.allclose(r, a, rtol=1e-6, atol=0), (net, r, a)


@pytest.mark.gpu
def test_all_ones_mask(nets):
    """vgg at 64x64: every tap size divides 64, so the all-ones masked LPIPS is LPIPS (up to float32 summation order).
    alex at 64x64: it is not."""
    from rodygs_b200.metrics import lpips, masked_lpips
    g = torch.Generator(device="cuda").manual_seed(4)
    x = torch.rand(2, 3, 64, 64, device="cuda", generator=g)
    y = (x + 0.1 * torch.randn(x.shape, device="cuda", generator=g)).clamp(0, 1)
    ones = torch.ones(2, 1, 64, 64, device="cuda")
    vgg, alex = nets["vgg"][0], nets["alex"][0]
    got, ref = masked_lpips(x, y, ones, vgg), lpips(x, y, vgg)
    assert torch.allclose(got, ref, rtol=2e-6, atol=0), (got, ref)
    y_edge = torch.cat([x[..., :-6], y[..., -6:]], -1)      # as in test_twin_closed_forms
    got, ref = masked_lpips(x, y_edge, ones, alex), lpips(x, y_edge, alex)
    assert ((got - ref).abs() / ref).min().item() > 1e-4, (got, ref)


@pytest.mark.gpu
def test_vgg_past_a_2_gib_workspace(nets):
    """vgg at 1200x1920 needs 2.36 GB of workspace: both calls run and are reproducible there."""
    from rodygs_b200.metrics import lpips, masked_lpips
    g = torch.Generator(device="cuda").manual_seed(6)
    x = torch.rand(3, 1200, 1920, device="cuda", generator=g)
    y = (x + 0.1 * torch.randn(x.shape, device="cuda", generator=g)).clamp(0, 1)
    m = covisibility_mask(1, 1200, 1920, g, "cuda")[0]
    w = nets["vgg"][0]
    a, b = lpips(x, y, w), masked_lpips(x, y, m, w)
    assert torch.isfinite(a).all() and (a > 0).all() and torch.isfinite(b).all() and (b > 0).all(), (a, b)
    assert torch.equal(lpips(x, y, w), a) and torch.equal(masked_lpips(x, y, m, w), b)
    assert torch.equal(masked_lpips(x, x, m, w), torch.zeros(1, device="cuda"))


def _table(step, views, gts, **kw):
    cams, vms, pms, bts = views
    return step.evaluate(vms, pms, [c.tanfovx for c in cams], cams[0].tanfovy, bts, gts, **kw)


@pytest.mark.gpu
def test_evaluate_adds_the_masked_lpips_columns(nets):
    from rodygs_b200.metrics import masked_lpips
    step = _make_step(20_000, 176, 208)
    views = _views(step, 3)
    gts = torch.rand(3, 3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4))
    masks = covisibility_mask(3, 176, 208, torch.Generator(device="cuda").manual_seed(5), "cuda")
    alex, vgg = nets["alex"][0], nets["vgg"][0]
    base = _table(step, views, gts, masks=masks, lpips=(alex, vgg))
    full = _table(step, views, gts, masks=masks, lpips=(alex, vgg), masked_lpips=alex)
    both = _table(step, views, gts, masks=masks, masked_lpips=[alex, vgg])
    assert base.shape == (3, 9) and full.shape == (3, 10) and both.shape == (3, 9)
    assert torch.equal(full[:, :9], base) and torch.equal(both[:, :7], base[:, :7])
    cams, vms, pms, bts = views
    for v, cam in enumerate(cams):
        color = _render(step, cam, vms[v], pms[v], bts[v])
        ra, rv = masked_lpips(color, gts[v], masks[v], alex), masked_lpips(color, gts[v], masks[v], vgg)
        assert torch.equal(full[v, 9:], ra), (v, full[v], ra)
        assert torch.equal(both[v, 7:], torch.cat([ra, rv])), (v, both[v], ra, rv)
    assert torch.isfinite(full).all() and torch.isfinite(both).all()
    with pytest.raises(ValueError, match="pass masks"):
        _table(step, views, gts, masked_lpips=alex)
    with pytest.raises(ValueError, match="masked_lpips must be"):
        _table(step, views, gts, masks=masks, masked_lpips=("alex",))


@pytest.mark.gpu
def test_evaluate_with_masked_lpips_leaves_the_training_state_alone(nets):
    """As test_gpu_metrics.test_evaluate_leaves_the_training_state_alone, with the masked LPIPS column."""
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
    masks = covisibility_mask(3, 176, 208, g, "cuda")
    for it in (1, 2):
        step.forward_backward(vms[0], pms[0], cams[0].tanfovx, cams[0].tanfovy, bts[0], gt, None, dcolor_slot=0)
        step.exchange_grads(vms[:1].contiguous(), bts[:1].contiguous(), defer_sh=True)
        if it == 1:
            for tag in ("static", "dynamic"):
                step.add_densification_stats(tag)
                step.optimizer_step(tag, it)
    torch.cuda.synchronize()
    before = _snapshot(step)
    table = step.evaluate(vms, pms, cams[0].tanfovx, cams[0].tanfovy, bts, gts, masks=masks, masked_lpips=nets["alex"][0])
    torch.cuda.synchronize()
    after = _snapshot(step)
    assert table.shape == (3, 8) and torch.isfinite(table).all()
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
    from rodygs_b200.metrics import load_lpips
    alex, vgg = (load_lpips(net, *random_weights(net, 50 + k)) for k, net in enumerate(("alex", "vgg")))
    step = _make_step(12_000, 176, 208)
    views = _views(step, 3)
    gts = torch.rand(3, 3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
    masks = covisibility_mask(3, 176, 208, torch.Generator(device="cuda").manual_seed(9), "cuda")
    return _table(step, views, gts, masks=masks, lpips=vgg, masked_lpips=(alex, vgg))


@pytest.mark.gpu
def test_evaluate_with_masked_lpips_on_two_ranks_matches_one_process():
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
    assert a.shape == (3, 10)
    assert torch.equal(a, b), (a, b)
    assert torch.equal(a, single), (a, single)
