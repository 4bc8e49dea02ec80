"""LPIPS on the device (rdg_lpips, rodygs_b200.metrics.load_lpips / lpips) and SplatTrainStep.evaluate(lpips=).

The reference is a float64 twin of the lpips package's definition as INTEGRATION.md "Scoring held-out views" states it,
written with F.conv2d, F.max_pool2d and the channel normalisation.  Weights are random (He-normal convs, small biases,
non-negative heads) under the real key names of the torchvision backbones and the lpips heads, so nothing is downloaded.
The twin can round each conv's operands to TF32 exactly as the kernel does (cvt.rna: to nearest, ties away from zero);
against that the kernel must agree to 1e-4 relative, and against the plain float64 twin (the cost of TF32) to 5e-3."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from test_gpu_metrics import _make_step, _render, _same, _snapshot, _views
from test_gpu_masked_metrics import covisibility_mask

from rodygs_b200.metrics import LPIPS_CONVS, LPIPS_TAPS

POOLS = {"alex": {3: 3, 6: 3}, "vgg": {5: 2, 10: 2, 17: 2, 24: 2}}     # features.{i} -> kernel of the stride-2 max-pool before it
TAPS = {"alex": (0, 3, 6, 8, 10), "vgg": (2, 7, 14, 21, 28)}
GEOM = {"alex": {0: (4, 2), 3: (1, 2)}}                                # (stride, padding) where not (1, 1)


# ================================================================ twin ==

def random_weights(net, seed):
    """(backbone state dict, linear state dict) with the real keys and shapes, float32 on the CPU."""
    g = torch.Generator().manual_seed(seed)
    bb = {}
    for i, cout, cin, k in LPIPS_CONVS[net]:
        bb[f"features.{i}.weight"] = torch.randn(cout, cin, k, k, generator=g) * (2.0 / (cin * k * k)) ** 0.5
        bb[f"features.{i}.bias"] = torch.randn(cout, generator=g) * 0.01
    bb["classifier.1.weight"] = torch.randn(16, 8, generator=g)        # ignored by the loader
    lin = {f"lin{l}.model.1.weight": torch.rand(1, c, 1, 1, generator=g) * 0.2 for l, c in enumerate(LPIPS_TAPS[net])}
    return bb, lin


def rna_tf32(t):
    """float32 rounding, then TF32 round-to-nearest, ties away from zero (cvt.rna.tf32.f32); returned in float64."""
    u = t.to(torch.float32).contiguous().view(torch.int32)
    return ((u + 0x1000) & ~0x1FFF).view(torch.float32).to(torch.float64)


def twin(pred, gt, bb, lin, net, value_range=1.0, tf32=False):
    """[B] LPIPS in float64 on the device of the inputs; pred, gt [B, 3, H, W]."""
    dev = pred.device
    mu = torch.tensor([0.485, 0.456, 0.406], dtype=torch.float64, device=dev).view(1, 3, 1, 1)
    sd = torch.tensor([0.229, 0.224, 0.225], dtype=torch.float64, device=dev).view(1, 3, 1, 1)
    z = (torch.cat([pred, gt]).double() / value_range - mu) / sd
    B = pred.shape[0]
    total = torch.zeros(B, dtype=torch.float64, device=dev)
    t = 0
    for i, _, _, _ in LPIPS_CONVS[net]:
        if i in POOLS[net]:
            z = F.max_pool2d(z, POOLS[net][i], 2)
        w = bb[f"features.{i}.weight"].to(dev, torch.float64)
        b = bb[f"features.{i}.bias"].to(dev, torch.float64)
        s, p = GEOM.get(net, {}).get(i, (1, 1))
        z = F.relu(F.conv2d(rna_tf32(z) if tf32 else z, rna_tf32(w) if tf32 else w, b, stride=s, padding=p))
        if i in TAPS[net]:
            n = z / (z.pow(2).sum(1, keepdim=True).sqrt() + 1e-10)
            wl = lin[f"lin{t}.model.1.weight"].to(dev, torch.float64)
            total += (wl * (n[:B] - n[B:]) ** 2).sum(1).mean((1, 2))
            t += 1
    return total


# ================================================================ CPU ==

def test_twin_of_identical_images_is_zero_and_shapes_are_the_torchvision_ones():
    for net in ("alex", "vgg"):
        bb, lin = random_weights(net, 0)
        x = torch.rand(1, 3, 40, 48, dtype=torch.float64)
        assert twin(x, x, bb, lin, net).item() == 0.0
        assert twin(x, x.flip(-1), bb, lin, net).item() > 0.0
    # the conv indices are those of torchvision's alexnet / vgg16 features
    assert [i for i, *_ in LPIPS_CONVS["alex"]] == [0, 3, 6, 8, 10]
    assert [i for i, *_ in LPIPS_CONVS["vgg"]] == [0, 2, 5, 7, 10, 12, 14, 17, 19, 21, 24, 26, 28]


def test_rna_tf32_rounds_to_nearest_ties_away():
    one = 1.0
    ulp = 2.0 ** -10                                      # TF32 keeps 10 mantissa bits
    x = torch.tensor([one + ulp * 0.5, one + ulp * 0.49, -(one + ulp * 0.5), one + ulp * 1.5], dtype=torch.float64)
    assert rna_tf32(x).tolist() == [one + ulp, one, -(one + ulp), one + 2 * ulp]


def test_loader_refuses_missing_keys_wrong_shapes_and_unknown_nets():
    from rodygs_b200.metrics import load_lpips
    bb, lin = random_weights("alex", 1)
    with pytest.raises(ValueError, match="net must be"):
        load_lpips("squeeze", bb, lin)
    for key in ("features.6.weight", "features.10.bias"):
        broken = {k: v for k, v in bb.items() if k != key}
        with pytest.raises(ValueError, match=f"missing key '{key}'"):
            load_lpips("alex", broken, lin)
    with pytest.raises(ValueError, match="missing key 'lin4.model.1.weight'"):
        load_lpips("alex", bb, {k: v for k, v in lin.items() if not k.startswith("lin4")})
    with pytest.raises(ValueError, match="'features.3.weight' must have shape"):
        load_lpips("alex", {**bb, "features.3.weight": torch.zeros(192, 64, 3, 3)}, lin)
    with pytest.raises(ValueError, match="'lin1.model.1.weight' must have shape"):
        load_lpips("alex", bb, {**lin, "lin1.model.1.weight": torch.zeros(1, 128, 1, 1)})
    vbb, vlin = random_weights("vgg", 1)
    with pytest.raises(ValueError, match="missing key 'features.28.weight'"):     # alex's keys are not vgg's
        load_lpips("vgg", {**bb, **{k: v for k, v in vbb.items() if k != "features.28.weight"}}, vlin)


def test_a_saved_state_dict_loads_like_the_in_memory_one(tmp_path):
    from rodygs_b200.metrics import load_lpips
    bb, lin = random_weights("vgg", 2)
    torch.save(bb, tmp_path / "vgg16.pth")
    torch.save(lin, tmp_path / "vgg.pth")
    broken = dict(lin)
    del broken["lin2.model.1.weight"]
    torch.save(broken, tmp_path / "broken.pth")
    with pytest.raises(ValueError, match="missing key 'lin2.model.1.weight'"):
        load_lpips("vgg", tmp_path / "vgg16.pth", tmp_path / "broken.pth")
    if torch.cuda.is_available():
        a = load_lpips("vgg", str(tmp_path / "vgg16.pth"), tmp_path / "vgg.pth")
        b = load_lpips("vgg", bb, lin)
        assert a.net == b.net == "vgg" and torch.equal(a.packed, b.packed)
    else:
        for src in ((str(tmp_path / "vgg16.pth"), tmp_path / "vgg.pth"), (bb, lin)):
            with pytest.raises(RuntimeError, match="no CPU fallback"):      # every key checked, then the device refused
                load_lpips("vgg", *src, device="cpu")


def test_lpips_refuses_cpu_tensors_channels_and_small_sizes():
    from rodygs_b200.metrics import LpipsWeights, lpips
    for net, edge in (("alex", 31), ("vgg", 16)):
        w = LpipsWeights(net, torch.zeros(1))
        with pytest.raises(RuntimeError, match="pred is on cpu"):
            lpips(torch.rand(3, 40, 40), torch.rand(3, 40, 40), w)
        with pytest.raises(ValueError, match="3 channels"):
            lpips(torch.rand(2, 4, 40, 40), torch.rand(2, 4, 40, 40), w)
        with pytest.raises(ValueError, match=f">= {edge}"):
            lpips(torch.rand(3, edge - 1, 64), torch.rand(3, edge - 1, 64), w)
        with pytest.raises(ValueError, match=f">= {edge}"):
            lpips(torch.rand(1, 3, 64, edge - 1), torch.rand(1, 3, 64, edge - 1), w)
    with pytest.raises(TypeError, match="LpipsWeights"):
        lpips(torch.rand(3, 40, 40), torch.rand(3, 40, 40), None)


def test_abi_refuses_bad_arguments_without_a_gpu():
    from rodygs_b200 import _lib
    lib = _lib.load()
    one = (C.c_float * 4)()
    alex, vgg = 0, 1
    n_alex, n_vgg = lib.rdg_lpips_packed_floats(alex), lib.rdg_lpips_packed_floats(vgg)
    assert n_alex > 2_400_000 and n_vgg > 14_700_000     # at least the conv weights of each backbone
    assert lib.rdg_lpips_packed_floats(2) == -1 and b"net" in lib.rdg_last_error()
    ws = lib.rdg_lpips_workspace_bytes(vgg, 64, 80)
    assert ws > 2 * 2 * 64 * 80 * 64 * 4
    for args, word in (((2, 64, 64), b"net"), ((alex, 30, 64), b"height"), ((alex, 64, 30), b"width"),
                       ((vgg, 15, 64), b"height"), ((vgg, 64, 15), b"width")):
        assert lib.rdg_lpips_workspace_bytes(*args) == -1
        assert word in lib.rdg_last_error()
    assert lib.rdg_lpips_workspace_bytes(alex, 31, 31) > 0 and lib.rdg_lpips_workspace_bytes(vgg, 16, 16) > 0

    def call(pred=one, gt=one, B=2, Cc=3, H=64, W=80, vr=1.0, net=vgg, packed=one, nf=n_vgg, out=one, w=one, nb=ws):
        return lib.rdg_lpips(pred, gt, B, Cc, H, W, vr, net, packed, nf, out, w, nb, None)

    for kw, word in ((dict(pred=None), b"pred"), (dict(gt=None), b"gt"), (dict(packed=None), b"packed"),
                     (dict(out=None), b"out"), (dict(w=None), b"workspace"), (dict(net=5), b"net"), (dict(B=0), b"batch"),
                     (dict(Cc=1), b"channels"), (dict(Cc=4), b"channels"), (dict(H=15), b"height"), (dict(W=15), b"width"),
                     (dict(vr=0.0), b"value_range"), (dict(vr=float("nan")), b"value_range"),
                     (dict(nf=n_vgg - 1), b"packed_floats"), (dict(nf=n_alex), b"packed_floats"),
                     (dict(nb=ws - 1), b"workspace_bytes")):
        assert call(**kw) == -1, kw
        assert word in lib.rdg_last_error(), (kw, lib.rdg_last_error())

    ptrs = lambda n, k=None: (C.c_void_p * n)(*[None if i == k else C.addressof(one) for i in range(n)])   # noqa: E731
    for net, nconv, nf in ((alex, 5, n_alex), (vgg, 13, n_vgg)):
        good = (ptrs(nconv), ptrs(nconv), ptrs(5))
        assert lib.rdg_lpips_pack(net, *good, one, nf - 1, None) == -1 and b"packed_floats" in lib.rdg_last_error()
        assert lib.rdg_lpips_pack(net, *good, None, nf, None) == -1 and b"packed" in lib.rdg_last_error()
        assert lib.rdg_lpips_pack(7, *good, one, nf, None) == -1 and b"net" in lib.rdg_last_error()
        for slot, word in ((0, b"conv_w"), (1, b"conv_b"), (2, b"lin_w")):
            arrs = list(good)
            assert lib.rdg_lpips_pack(net, *[None if j == slot else a for j, a in enumerate(arrs)], one, nf, None) == -1
            assert word in lib.rdg_last_error()
            arrs[slot] = ptrs(5 if slot == 2 else nconv, 3)
            assert lib.rdg_lpips_pack(net, *arrs, one, nf, None) == -1
            assert word + b"[3]" in lib.rdg_last_error()


# ================================================================ GPU ==

@pytest.fixture(scope="module")
def no_tf32():
    # the twins are float64; keep cuDNN from doing anything but exact float64 arithmetic either way
    saved = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32 = saved


@pytest.fixture(scope="module")
def nets():
    from rodygs_b200.metrics import load_lpips
    out = {}
    for k, net in enumerate(("alex", "vgg")):
        bb, lin = random_weights(net, 10 + k)
        out[net] = (load_lpips(net, bb, lin), bb, lin)
    return out


def _render_pair(H, W, n, seed):
    """A synthetic render against the same render plus noise, [1, 3, H, W] each."""
    step = _make_step(n, H, W)
    cams, vms, pms, bts = _views(step, 1)
    a = _render(step, cams[0], vms[0], pms[0], bts[0]).clone()[None]
    g = torch.Generator(device="cuda").manual_seed(seed)
    b = (a + 0.05 * torch.randn(a.shape, device="cuda", generator=g)).clamp(0, 1)
    return a, b


_ERR = {}


@pytest.mark.gpu
@pytest.mark.parametrize("net,H,W", [("alex", 64, 64), ("vgg", 64, 64), ("alex", 97, 131), ("vgg", 97, 131),
                                     ("alex", 1080, 1920), ("vgg", 540, 960)])
def test_kernel_against_the_twin(net, H, W, nets, no_tf32):
    """Layout bar: 1e-4 relative against the twin with the kernel's TF32 operand rounding.  Cost of TF32: 5e-3 relative
    against the plain float64 twin."""
    from rodygs_b200.metrics import lpips
    w, bb, lin = nets[net]
    pred, gt = _render_pair(H, W, 20_000 if H < 200 else 150_000, H + W)
    got = lpips(pred, gt, w).double()
    ref_tf32 = twin(pred, gt, bb, lin, net, tf32=True)
    ref64 = twin(pred, gt, bb, lin, net)
    layout = ((got - ref_tf32).abs() / ref_tf32.abs()).max().item()
    cost = ((got - ref64).abs() / ref64.abs()).max().item()
    print(f"\n{net} {H}x{W}: kernel {got.tolist()} tf32-twin {ref_tf32.tolist()} float64 {ref64.tolist()} "
          f"rel err vs tf32 twin {layout:.3e}, vs float64 {cost:.3e}")
    assert got.item() > 0
    assert layout <= 1e-4, (net, H, W, layout)
    assert cost <= 5e-3, (net, H, W, cost)


@pytest.mark.gpu
def test_exact_properties(nets):
    from rodygs_b200.metrics import lpips
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.rand(3, 3, 70, 90, device="cuda", generator=g)
    y = (x + 0.1 * torch.randn(x.shape, device="cuda", generator=g)).clamp(0, 1)
    for net in ("alex", "vgg"):
        w = nets[net][0]
        assert torch.equal(lpips(x, x, w), torch.zeros(3, device="cuda"))
        a, b = lpips(x, y, w), lpips(x, y, w)
        assert torch.equal(a, b)
        assert a.shape == (3,) and a.dtype == torch.float32 and (a > 0).all()
        for i in range(3):
            assert torch.equal(lpips(x[i], y[i], w), a[i:i + 1])
        r = lpips(255 * x, 255 * y, w, value_range=255)
        assert torch.allclose(r, a, rtol=1e-6, atol=0), (net, r, a)
        assert torch.equal(lpips(x.double(), y.half().float(), w), lpips(x, y.half().float(), w))   # dtypes convert


def _table(step, views, gts, **kw):
    cams, vms, pms, bts = views
    return step.evaluate(vms, pms, [c.tanfovx for c in cams], cams[0].tanfovy, bts, gts, **kw)


@pytest.mark.gpu
def test_evaluate_adds_the_lpips_columns(nets):
    from rodygs_b200.metrics import lpips
    step = _make_step(20_000, 176, 208)
    views = _views(step, 3)
    gts = torch.rand(3, 3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4))
    masks = covisibility_mask(3, 176, 208, torch.Generator(device="cuda").manual_seed(5), "cuda")
    alex, vgg = nets["alex"][0], nets["vgg"][0]
    plain = _table(step, views, gts)
    masked = _table(step, views, gts, masks=masks)
    both = _table(step, views, gts, lpips=(alex, vgg))
    one = _table(step, views, gts, lpips=vgg)
    full = _table(step, views, gts, masks=masks, lpips=[alex, vgg])
    assert both.shape == (3, 6) and one.shape == (3, 5) and full.shape == (3, 9)
    assert torch.equal(both[:, :4], plain) and torch.equal(one[:, :4], plain) and torch.equal(full[:, :7], masked)
    cams, vms, pms, bts = views
    for v, cam in enumerate(cams):
        color = _render(step, cam, vms[v], pms[v], bts[v])
        ra, rv = lpips(color, gts[v], alex), lpips(color, gts[v], vgg)
        assert torch.equal(both[v, 4:], torch.cat([ra, rv])), (v, both[v], ra, rv)
        assert torch.equal(full[v, 7:], both[v, 4:]) and torch.equal(one[v, 4:], rv)
    assert torch.isfinite(full).all()
    with pytest.raises(ValueError, match="lpips must be"):
        _table(step, views, gts, lpips=("alex",))


@pytest.mark.gpu
def test_evaluate_with_lpips_leaves_the_training_state_alone(nets):
    """As test_gpu_metrics.test_evaluate_leaves_the_training_state_alone, with both LPIPS columns."""
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
    table = step.evaluate(vms, pms, cams[0].tanfovx, cams[0].tanfovy, bts, gts, lpips=(nets["alex"][0], nets["vgg"][0]))
    torch.cuda.synchronize()
    after = _snapshot(step)
    assert table.shape == (3, 6) and torch.isfinite(table).all()
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
    ws = [load_lpips(net, *random_weights(net, 20 + k)) for k, net in enumerate(("alex", "vgg"))]
    step = _make_step(12_000, 176, 208)
    views = _views(step, 3)
    gts = torch.rand(3, 3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
    return _table(step, views, gts, lpips=ws)


@pytest.mark.gpu
def test_evaluate_with_lpips_on_two_ranks_matches_one_process():
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
    assert a.shape == (3, 6)
    assert torch.equal(a, b), (a, b)
    assert torch.equal(a, single), (a, single)


def test_conv_kernel_runs_on_the_tensor_cores():
    """The conv kernel's SASS issues tcgen05.mma (UTCHMMA) and tcgen05.ld (LDTM), has no FFMA main loop, and spills
    nothing."""
    import os
    import shutil
    import subprocess
    import tempfile
    from rodygs_b200 import build
    nvcc, cuobjdump = build._nvcc(), shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "lpips.o")
        r = subprocess.run([nvcc, *build.ARCH, *build.COMMON, "-Xptxas", "-v", "-c", os.path.join(build.CSRC, "lpips.cu"),
                            "-o", obj], capture_output=True, text=True, check=True)
        assert "spill" in r.stderr and all(" 0 bytes spill stores, 0 bytes spill loads" in line
                                           for line in r.stderr.splitlines() if "spill" in line), r.stderr
        sass = subprocess.run([cuobjdump, "-sass", "-fun", "_Z17lpips_conv_kernel6LpConv", obj], capture_output=True,
                              text=True, check=True).stdout
    assert "UTCHMMA" in sass and "LDTM" in sass
    assert "FFMA" not in sass
