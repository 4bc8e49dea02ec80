"""The kernels that PRODUCE gradients - the loss stage that seeds the rasterizer backward, the motion regularisers that add
into the flat gradient buffer, rigidity, the sample gather / scatter and the basis MLP backward - element-wise against
float64, at production shapes and at the edges where they can go wrong.

The references are float64 twins written with plain torch ops that follow the device and dtype of their inputs, so they
run on the GPU (the oracle package builds its SSIM taps and identity matrices on the CPU, and float64 photometric loss
and backward at 3x1080x1920 takes ~20 s there).  Each twin is pinned to its oracle function on the CPU (part 1).
Discrete choices the kernel makes are inputs of the reference: rigidity takes the neighbour indices `knn_points` gave the
kernel and recomputes their squared distances in float64, so the chain through dist2 is differentiated.

Bar, per element (helpers.elementwise_vs_truth): |a - b64| <= 1e-3 |b64| + 1e-5 max|b64|, or 1.5 x the error of the same
twin run in float32 on the GPU where float32 cannot resolve the float64 value.  Loss values: 2e-6 relative to float64,
or 1.5 x the float32 twin's own error.  Exact where the math is exact (dL/dalpha, L1 at ties, all-zero coefficient rows,
gradient entries a kernel must leave alone).  test_elementwise_bar_rejects_plausible_kernel_bugs (CPU) shows that the bar
catches five plausible kernel bugs on the cases meant to catch them, and which of them the norm-wise bar would accept."""
import copy
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

import helpers
from oracle import deform_oracle as do
from oracle import loss_oracle as lo
from oracle import motion_oracle as mo

CUDA = "cuda"
EPS = 1e-6
W4 = dict(w_l1=0.8, w_dssim=0.2, w_pearson=0.05, w_local=0.15, w_alpha=0.01)   # config 4 loss weights
WORST = {}                                                                      # kernel -> (r_cu, r_32, check)
WORST_VALUE = [0.0, ""]                                                         # loss values: |a - b64| / (2e-6 |b64|)


@pytest.fixture(scope="module", autouse=True)
def _report():
    # the float32 twins set the allowance where float32 cannot resolve float64: they must not run in TF32
    tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    if torch.cuda.is_available():
        torch.cuda.reset_peak_memory_stats()
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    if WORST:
        print("\nworst element-wise ratio per kernel (r_cu / r_32 = CUDA / float32 twin, vs float64; bar 1.0):")
        for k, (rc, r3, name) in sorted(WORST.items()):
            print(f"  {k:28s} r_cu {rc:.3f}  r_32 {r3:.3f}  ({name})")
    if WORST_VALUE[1]:
        print(f"worst loss value: {WORST_VALUE[0]:.3f} x 2e-6 relative ({WORST_VALUE[1]})")
    if torch.cuda.is_available():
        print(f"peak device memory: {torch.cuda.max_memory_allocated() / 2**30:.2f} GiB")


def _bar(kernel, name, got, ref32, ref64, mask=None):
    if mask is not None:
        got, ref32, ref64 = got[mask], ref32[mask], ref64[mask]
    ok, r_cu, r_32 = helpers.elementwise_vs_truth(got, ref32, ref64)
    if kernel not in WORST or r_cu > WORST[kernel][0] or r_cu != r_cu:
        WORST[kernel] = (r_cu, r_32, name)
    assert ok, f"{kernel} {name}: element-wise {r_cu:.3f} x (1e-3 |b| + 1e-5 max|b|) vs float64 (float32 twin {r_32:.3f} x)"


def _value(name, got, v64, rtol=2e-6):
    got, v64 = float(got), float(v64)
    r = abs(got - v64) / (rtol * abs(v64))
    if r > WORST_VALUE[0]:
        WORST_VALUE[:] = [r, name]
    assert r <= 1.0, f"{name}: {got!r} vs float64 {v64!r}: {r:.2f} x 2e-6 relative"


# ================================================================ twins (device-agnostic) ==

def _blur(x, taps):
    """Separable 11-tap Gaussian blur of [C,H,W], zero padding 5, per channel."""
    ch = x.shape[0]
    y = F.conv2d(x[None], taps.view(1, 1, 1, -1).expand(ch, 1, 1, 11), padding=(0, 5), groups=ch)
    return F.conv2d(y, taps.view(1, 1, -1, 1).expand(ch, 1, 11, 1), padding=(5, 0), groups=ch)[0]


def ssim_map(a, b):
    t = lo.gauss_taps(a.dtype).to(a.device)
    mu1, mu2 = _blur(a, t), _blur(b, t)
    mu1_sq, mu2_sq, mu12 = mu1 * mu1, mu2 * mu2, mu1 * mu2
    s1, s2, s12 = _blur(a * a, t) - mu1_sq, _blur(b * b, t) - mu2_sq, _blur(a * b, t) - mu12
    return ((2 * mu12 + lo.SSIM_C1) * (2 * s12 + lo.SSIM_C2)) / ((mu1_sq + mu2_sq + lo.SSIM_C1) * (s1 + s2 + lo.SSIM_C2))


def photometric(pred, gt, w_l1=0.8, w_dssim=0.2):
    """(loss, l1, ssim)."""
    l1 = (pred - gt).abs().mean()
    s = ssim_map(pred, gt).mean()
    return w_l1 * l1 + w_dssim * (1.0 - s), l1, s


def pearson(p, g, eps=EPS):
    p, g = p.reshape(-1), g.reshape(-1)
    pc, gc = p - p.mean(), g - g.mean()
    return 1.0 - ((pc / (pc.std() + eps)) * (gc / (gc.std() + eps))).mean()


def pearson_boxes(p, g, boxes, eps=EPS):
    """[n_boxes] Pearson losses over (row0, col0, rows, cols) boxes of [.., H, W] maps."""
    return torch.stack([pearson(p[..., r:r + h, c:c + w], g[..., r:r + h, c:c + w], eps) for r, c, h, w in boxes])


def alpha_term(alpha, w_alpha):
    return w_alpha * (1.0 - alpha).mean()


def _first_argmax(a):
    """Index of the first maximum along the last dim (torch.max's choice on the CPU), never device-dependent."""
    mx = a.max(dim=-1, keepdim=True).values
    ar = torch.arange(a.shape[-1], device=a.device)
    return torch.where(a == mx, ar, a.shape[-1]).min(dim=-1, keepdim=True).values


def motion_l1(c):
    return c.abs().mean()


def motion_sparsity(c):
    a = c.abs()
    mx = a.gather(-1, _first_argmax(a.detach()))
    return (a / (mx + 1e-7)).mean()


def quat_to_matrix(q):
    r, i, j, k = torch.unbind(q, -1)
    two_s = 2.0 / (q * q).sum(-1)
    o = torch.stack((1 - two_s * (j * j + k * k), two_s * (i * j - k * r), two_s * (i * k + j * r),
                     two_s * (i * j + k * r), 1 - two_s * (i * i + k * k), two_s * (j * k - i * r),
                     two_s * (i * k - j * r), two_s * (j * k + i * r), 1 - two_s * (i * i + j * j)), -1)
    return o.reshape(q.shape[:-1] + (3, 3))


def motion_basis_reg(table, reg, td=0, rd=0):
    """(translation term, rotation term, loss) of MotionBasisRegularizaiton at degree 0 (negative: off)."""
    R = quat_to_matrix(table[..., 3:])
    dtr, dR = table[1:, :, :3] - table[:-1, :, :3], R[1:] - R[:-1]
    eye = torch.eye(3, dtype=table.dtype, device=table.device)
    t = (torch.norm(dtr, dim=-1) * reg).mean()
    r = (torch.norm(eye - dR, dim=(-1, -2)) * reg).mean()
    return t, r, (t if td >= 0 else 0.0) + (r if rd >= 0 else 0.0)


def rigidity(points, canon, coeff, table, fi, nn, surface=True, distance=True, eps=EPS, drop_nb_from=None):
    """(surface, distance_preserving) of RigidityLoss for the neighbour indices nn [n, K]; coeff [n, B].
    drop_nb_from=k: the neighbour's half of the distance force is dropped for k >= that (a mutant for the bar test)."""
    nnl = nn.long()
    zero = points.new_zeros(())
    s = d = zero
    if surface:
        s = F.pairwise_distance(points, points[nnl].mean(dim=1), p=2).mean()
    if distance:
        n, K, Ts = nnl.shape[0], nnl.shape[1], fi.numel()
        diff = points[:, None] - points[nnl]
        dd = (diff[..., 0] * diff[..., 0] + diff[..., 1] * diff[..., 1]) + diff[..., 2] * diff[..., 2]    # [n, K]
        B3 = table[fi.long()][..., :3]                                                                 # [Ts, B, 3]
        loc = canon[None] + torch.einsum("nb,tbd->tnd", coeff, B3)                                     # [Ts, n, 3]
        loc_nn = loc[:, nnl]                                                                           # [Ts, n, K, 3]
        if drop_nb_from is not None:
            loc_nn = torch.cat((loc_nn[:, :, :drop_nb_from], loc_nn[:, :, drop_nb_from:].detach()), 2)
        x = torch.norm(loc_nn - loc[:, :, None], dim=-1)                                               # [Ts, n, K]
        # the reference pairs flat element f of the [Ts, n, K] block with neighbour distance f / Ts (a .view, kept)
        xv, yv = x.contiguous().view(-1, Ts, 1), dd.reshape(-1, 1, 1)
        d = torch.sqrt((xv - yv).pow(2) + eps ** 2).sum() / (n * K * Ts)
    return s, d


def sample_points(xyz, coeff, table, bt, time_ind, idx, lr):
    """xyz[i] + lr * sum_b c_ib (B(t) - table[t_i])_b[:3] for the sampled rows i (rodygs_dynamic.py:122-138)."""
    c = coeff[idx]
    delta = (c[:, :, None] * (bt[None, :, :3] - table[time_ind[idx].long()][..., :3])).sum(1)
    return xyz[idx] + lr * delta


def _leaves(dtype, device, *ts):
    return [t.detach().to(device, dtype).clone().requires_grad_(True) for t in ts]


# ================================================================ part 1: twins pinned to the oracle (CPU) ==

def _close(a, b, dtype):
    # float32: the CPU reductions of torch split their sums over threads in an order that is not fixed, and the rigidity
    # pin sums ~1e4 terms (float32 error ~ sqrt(N) eps ~ 1e-5 relative), so 2e-5 left no margin
    tol = 1e-12 if dtype == torch.float64 else 1e-4
    return helpers.rel_err(a.detach(), b.detach()) <= tol


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_photometric_twin_matches_oracle(dtype):
    g = torch.Generator().manual_seed(1)
    a = torch.rand(3, 37, 45, generator=g)
    b = (a + 0.2 * torch.randn(3, 37, 45, generator=g)).clamp(0, 1)
    b[:, :5] = a[:, :5]
    x, y = _leaves(dtype, "cpu", a, a)
    bb = b.to(dtype)
    ref = lo.photometric(x, bb)
    got, l1, s = photometric(y, bb)
    assert _close(got, ref, dtype) and _close(l1, lo.l1(x, bb), dtype) and _close(s, lo.ssim(x, bb), dtype)
    assert _close(ssim_map(y, bb), lo.ssim_map(x, bb), dtype)
    (gr,) = torch.autograd.grad(ref, x)
    (gg,) = torch.autograd.grad(got, y)
    assert _close(gg, gr, dtype), helpers.rel_err(gg, gr)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_pearson_and_alpha_twins_match_oracle(dtype):
    g = torch.Generator().manual_seed(2)
    d1 = torch.rand(1, 60, 70, generator=g) * 5 + 1
    d2 = d1 * 0.7 + torch.rand(1, 60, 70, generator=g)
    d1[:, 10:18, 20:28] = 0.0                                         # an all-zero box: torch's masked std backward
    x, y = _leaves(dtype, "cpu", d1, d1)
    gt = d2.to(dtype)
    x0, y0 = torch.tensor([10, 3, 40, 0]), torch.tensor([20, 50, 40, 0])
    ref = lo.pearson_depth(x, gt) + lo.local_pearson_depth(x, gt, x0, y0, 8)
    boxes = [(r, c, 8, 8) for r, c in zip(x0.tolist(), y0.tolist())]
    got = pearson(y, gt) + pearson_boxes(y, gt, boxes).mean()
    assert _close(got, ref, dtype)
    (gr,) = torch.autograd.grad(ref, x)
    (gg,) = torch.autograd.grad(got, y)
    assert _close(gg, gr, dtype)
    assert gg[0, 10:18, 20:28].abs().max() > 1e3                      # ~ 1 / eps: the zero box's gradient
    # a rectangular box is the oracle's Pearson on that slice
    assert _close(pearson_boxes(y, gt, [(5, 9, 11, 37)])[0], lo.pearson_depth(x[:, 5:16, 9:46], gt[:, 5:16, 9:46]), dtype)
    al = torch.rand(1, 60, 70, generator=g).to(dtype)
    assert _close(alpha_term(al, 0.01), 0.01 * (1.0 - al).mean(), dtype)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_coefficient_twins_match_oracle_and_route_ties_to_the_first_index(dtype):
    g = torch.Generator().manual_seed(3)
    c = torch.randn(300, 1, 16, generator=g) * 0.2
    c[0] = 0.0
    c[1, 0, [2, 9]] = torch.tensor([0.7, -0.7])                       # c and -c: a two-way tie of max|c|
    c[2, 0, [1, 5, 6, 15]] = torch.tensor([0.9, -0.9, 0.9, 0.9])      # a four-way tie
    x, y = _leaves(dtype, "cpu", c, c)
    ref = 0.01 * mo.motion_l1(x) + 0.002 * mo.motion_sparsity(x)
    got = 0.01 * motion_l1(y) + 0.002 * motion_sparsity(y)
    assert _close(got, ref, dtype)
    (gr,) = torch.autograd.grad(ref, x)
    (gg,) = torch.autograd.grad(got, y)
    assert _close(gg, gr, dtype)
    # the oracle's torch.max sends the max term to the first index only: the other tied entries keep the plain gradient
    for row, first, others in ((1, 2, [9]), (2, 1, [5, 6, 15])):
        assert abs(gr[row, 0, first]) < abs(gr[row, 0, others[0]])
        for o in others[1:]:
            assert gr[row, 0, o].abs() == gr[row, 0, others[0]].abs()
    assert torch.equal(gr[0], torch.zeros_like(gr[0])) and torch.equal(gg[0], torch.zeros_like(gg[0]))


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("td,rd", [(0, 0), (0, -1), (-1, 0)])
def test_basis_reg_twin_matches_oracle(dtype, td, rd):
    g = torch.Generator().manual_seed(4)
    tb = _basis_table(12, g)
    reg = _reg("cum_exponential")
    x, y = _leaves(dtype, "cpu", tb, tb)
    ref = mo.motion_basis_reg(x, reg.to(dtype), td, rd)
    got = motion_basis_reg(y, reg.to(dtype), td, rd)[2]
    assert _close(got, ref, dtype)
    (gr,) = torch.autograd.grad(ref, x)
    (gg,) = torch.autograd.grad(got, y)
    assert _close(gg, gr, dtype)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("mode", [("distance_preserving", "surface"), ("surface",), ("distance_preserving",)])
def test_rigidity_twin_matches_oracle_for_given_neighbours(dtype, mode):
    g = torch.Generator().manual_seed(5)
    N, T, K = 700, 10, 8
    xyz = torch.randn(N, 3, generator=g)
    xyz[600:650] = xyz[:50]                                           # exact duplicates
    coeff = torch.randn(N, 1, 16, generator=g) * 0.2
    coeff[600:650] = coeff[:50]
    table = torch.randn(T, 16, 7, generator=g) * 0.1
    pred = torch.randn(N, 3, generator=g) * 0.02
    pred[600:650] = pred[:50]
    indice = torch.randperm(N, generator=g)[: N // 2]
    fi = torch.randint(0, T - 1, (5,), generator=g)
    ox, oc, ot, op = _leaves(dtype, "cpu", xyz, coeff, table, pred)
    ref, parts = mo.rigidity(ox, oc, torch.zeros(N, 1, 3, dtype=dtype), op, ot, indice, fi, K=K, mode=mode)
    tx, tc, tt, tp = _leaves(dtype, "cpu", xyz, coeff, table, pred)
    points = tx[indice] + tp[indice]
    _, nn = mo.knn_points(points.detach(), K)
    s, d = rigidity(points, tx[indice], tc.squeeze(1)[indice], tt, fi, nn, "surface" in mode, "distance_preserving" in mode)
    assert _close(s + d, ref, dtype)
    gr = torch.autograd.grad(ref, [ox, oc, ot, op], allow_unused=True)
    gg = torch.autograd.grad(s + d, [tx, tc, tt, tp], allow_unused=True)
    for a, b in zip(gg, gr):
        if b is None:
            assert a is None or a.abs().max() == 0
        else:
            assert _close(a, b, dtype), helpers.rel_err(a, b)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_sample_deformation_twin_matches_oracle(dtype):
    g = torch.Generator().manual_seed(6)
    nd, T = 500, 9
    xyz, coeff = torch.randn(nd, 3, generator=g), torch.randn(nd, 16, generator=g) * 0.1
    table, bt = torch.randn(T, 16, 7, generator=g) * 0.05, torch.randn(16, 7, generator=g) * 0.05
    ti = torch.randint(0, T, (nd,), generator=g)
    idx = torch.randperm(nd, generator=g)[:200]
    x = _leaves(dtype, "cpu", xyz, coeff, table, bt)
    y = _leaves(dtype, "cpu", xyz, coeff, table, bt)
    tr, _ = do.gaussian_deformation(x[1], x[3], x[2], ti, 1.7)
    ref = (x[0] + tr)[idx]
    got = sample_points(y[0], y[1], y[2], y[3], ti, idx, 1.7)
    assert _close(got, ref, dtype)
    up = torch.randn(200, 3, generator=g).to(dtype)
    for a, b in zip(torch.autograd.grad(got, y, up), torch.autograd.grad(ref, x, up)):
        assert _close(a, b, dtype)


def _reg(mode):
    from rodygs_b200 import motion_reg as mr
    return mr.basis_reg_coeff(mode)


def _basis_table(T, g, nb=16):
    """Rows with translations ~0.1 and non-unit quaternions |q| in [0.3, 3]; some rows repeat the frame before
    (zero translation change: torch.norm's zero sub-gradient)."""
    tb = torch.randn(T, nb, 7, generator=g) * 0.1
    q = torch.randn(T, nb, 4, generator=g)
    q = q / q.norm(dim=-1, keepdim=True) * (0.3 + 2.7 * torch.rand(T, nb, 1, generator=g))
    tb[..., 3:] = q
    for t in range(1, T, 4):
        tb[t, ::3] = tb[t - 1, ::3]
    return tb


# ================================================================ part 2: the bar has teeth (CPU) ==

def test_elementwise_bar_rejects_plausible_kernel_bugs():
    """Four plausible kernel bugs built on the float64 twins; the element-wise bar rejects each on the case meant to catch
    it.  Which of them the norm-wise bar max|a-b| / max|b| <= 1e-3 (the suite's old gradient bar) accepts is printed."""
    g = torch.Generator().manual_seed(7)
    f64 = torch.float64
    accepted = []

    def judge(name, mut, ref, mask=None):
        assert not torch.equal(mut, ref), name
        elem_ok = helpers.elementwise_ok(mut, ref)[0] if mask is None else helpers.elementwise_ok(mut[mask], ref[mask])[0]
        norm_ok = helpers.rel_err(mut, ref) <= 1e-3
        assert not elem_ok, f"the element-wise bar accepts the mutant '{name}'"
        if norm_ok:
            accepted.append(name)

    H, W = 97, 131
    d1 = (torch.rand(1, H, W, generator=g) * 5 + 1).to(f64)
    d2 = d1 * 0.7 + torch.rand(1, H, W, generator=g).to(f64)
    # (b) rows and cols swapped in a rectangular box (rdg_pearson)
    x = d1.clone().requires_grad_(True)
    rect = [(3, 5, 20, 90), (40, 7, 50, 30)]
    (ref,) = torch.autograd.grad(pearson_boxes(x, d2, rect).sum(), x)
    (mut,) = torch.autograd.grad(pearson_boxes(x, d2, [(r, c, w, h) for r, c, h, w in rect]).sum(), x)
    judge("rows and cols swapped in a rectangular box", mut, ref)
    # (c) the last partial row of 32x32 tiles (1080 = 33 * 32 + 24) skipped in SSIM pass 2: dL/dpred never written there
    a = torch.rand(3, 1080, 40, generator=g).to(f64)
    b = (a + 0.1 * torch.randn(3, 1080, 40, generator=g).to(f64)).clamp(0, 1)
    x = a.clone().requires_grad_(True)
    (ref,) = torch.autograd.grad(photometric(x, b)[0], x)
    mut = ref.clone()
    mut[:, 33 * 32:] = 0.0
    judge("last partial tile row skipped in SSIM pass 2", mut, ref)
    # (d) k2 unguarded at sp == 0: an all-zero depth box, the kernel's closed form with 0 / 0
    d = d1.clone()
    d[:, 20:36, 30:46] = 0.0
    x = d.clone().requires_grad_(True)
    (ref,) = torch.autograd.grad(pearson_boxes(x, d2, [(20, 30, 16, 16)]).sum(), x)
    for guard in (True, False):
        p, q = d[:, 20:36, 30:46].reshape(-1), d2[:, 20:36, 30:46].reshape(-1)
        m = p.numel()
        mp, mg = p.mean(), q.mean()
        sp, sg = (p - mp).pow(2).sum().div(m - 1).sqrt(), (q - mg).pow(2).sum().div(m - 1).sqrt()
        spg = ((p - mp) * (q - mg)).sum()
        k1 = 1.0 / (m * (sp + EPS) * (sg + EPS))
        k2 = spg / (m * (sp + EPS) ** 2 * (sg + EPS)) / ((m - 1) * sp) if (sp > 0 or not guard) else 0.0
        closed = torch.zeros_like(d)
        closed[:, 20:36, 30:46] = (-((q - mg) * k1 - (p - mp) * k2)).reshape(1, 16, 16)
        if guard:
            assert helpers.elementwise_ok(closed, ref, rtol=1e-12, floor=0)[0]     # the guarded form is torch's gradient
        else:
            judge("k2 unguarded at sp == 0", closed, ref)
    # (e) rigidity: the neighbour's half of the distance force dropped for k >= 8 (K = 16)
    n, K = 600, 16
    pts = torch.randn(n, 3, generator=g).to(f64)
    coeff = (torch.randn(n, 16, generator=g) * 0.2).to(f64)
    table = (torch.randn(12, 16, 7, generator=g) * 0.1).to(f64)
    fi = torch.randint(0, 11, (3,), generator=g)
    _, nn = mo.knn_points(pts, K)
    outs = []
    for drop in (None, 8):
        c, tb = coeff.clone().requires_grad_(True), table.clone().requires_grad_(True)
        _, dp = rigidity(pts, pts, c, tb, fi, nn, surface=False, drop_nb_from=drop)
        outs.append(torch.autograd.grad(dp, [c, tb]))
    judge("rigidity: neighbour half of the force dropped for k >= 8 (d_coeff)", outs[1][0], outs[0][0])
    print("accepted by the norm-wise bar:", accepted or "none")


def _depth_grad(d1, d2, boxes, n_boxes, w, dtype):
    """dL/ddepth of w_pearson * Pearson + w_local / n_boxes * sum over `boxes` of the box Pearson (CPU)."""
    x = d1.to(dtype).requires_grad_(True)
    gd = d2.to(dtype)
    loss = w["w_pearson"] * pearson(x, gd)
    if boxes:
        loss = loss + w["w_local"] / n_boxes * pearson_boxes(x, gd, boxes).sum()
    return torch.autograd.grad(loss, x)[0]


@pytest.mark.parametrize("H,W,s,n_boxes", [(1080, 1920, 128, 60), (97, 131, 16, 33), (33, 70, 16, 33)])
def test_depth_bar_rejects_pass2_bugs_on_the_loss_cases(H, W, s, n_boxes):
    """Bugs of the loss stage's pass 2 that leave the forward box sums (out[5]) intact, built on the inputs and boxes of
    test_loss_stage_against_float64 and judged the way it judges dL/ddepth (zero box, flat box and the rest of the map
    each against its own max): every one is rejected.  The norm-wise bar on the whole map accepts those printed."""
    _, _, d1, d2, _, boxes, special = _loss_inputs(H, W, s, n_boxes, 100 + H)
    g64 = _depth_grad(d1, d2, boxes, n_boxes, W4, torch.float64)
    g32 = _depth_grad(d1, d2, boxes, n_boxes, W4, torch.float32)
    regions = _depth_regions(H, W, special, "cpu")
    mutants = {}
    if H % 32:
        m = g64.clone()
        m[:, 32 * (H // 32):] = 0.0
        mutants["last partial tile row not written"] = m
    if W % 32:
        m = g64.clone()
        m[:, :, 32 * (W // 32):] = 0.0
        mutants["last partial tile column not written"] = m
    for flush in ((H - s, W - s, s, s), (H - s, 0, s, s)):
        mutants[f"flush box {flush[:2]} dropped"] = _depth_grad(d1, d2, [b for b in boxes if b != flush], n_boxes, W4,
                                                                torch.float64)
    mutants["boxes from the 33rd on dropped"] = _depth_grad(d1, d2, boxes[:32], n_boxes, W4, torch.float64)
    m = g64 * 1.25
    m[regions[1][1]] = g64[regions[1][1]]
    mutants["every entry outside the flat box x 1.25"] = m
    accepted = []
    for name, mut in mutants.items():
        assert not torch.equal(mut, g64), name
        assert not all(helpers.elementwise_vs_truth(mut[r], g32[r], g64[r])[0] for _, r in regions), \
            f"{H}x{W}: the element-wise bar accepts the mutant '{name}'"
        if helpers.rel_err(mut, g64) <= 1e-3:
            accepted.append(name)
    # and it accepts the float32 twin itself
    assert all(helpers.elementwise_vs_truth(g32[r], g32[r], g64[r])[0] for _, r in regions)
    print(f"{H}x{W}: accepted by the norm-wise bar:", accepted or "none")


# ================================================================ part 3: the loss stage (GPU) ==

def _loss_stage(pred, gt, depth, gtd, alpha, boxes, w):
    """rdg_losses through the C ABI, as SplatTrainStep calls it; untouched outputs keep their fill (-1 / 7)."""
    from rodygs_b200 import _lib
    lib = _lib.load()
    ch, H, W = pred.shape
    out = torch.full((8,), -1.0, device=CUDA)
    gcol = torch.full_like(pred, 7.0)
    gdep = torch.full((1, H, W), 7.0, device=CUDA)
    galp = torch.full((1, H, W), 7.0, device=CUDA)
    ws_bytes = int(lib.rdg_l1_dssim_workspace_bytes(ch, H, W))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=CUDA)
    terms = _lib.RdgLossTerms()
    terms.depth, terms.gt_depth, terms.dL_ddepth = depth.data_ptr(), gtd.data_ptr(), gdep.data_ptr()
    terms.w_pearson, terms.pearson_eps = w["w_pearson"], EPS
    terms.alpha, terms.dL_dalpha, terms.w_alpha = alpha.data_ptr(), galp.data_ptr(), w["w_alpha"]
    bx = None
    if boxes:
        bx = torch.tensor(boxes, dtype=torch.int32, device=CUDA).contiguous()
        terms.local_boxes, terms.n_local_boxes, terms.w_local = bx.data_ptr(), len(boxes), w["w_local"]
    _lib.check(lib.rdg_losses(pred.data_ptr(), gt.data_ptr(), ch, H, W, w["w_l1"], w["w_dssim"], C.byref(terms),
                              out.data_ptr(), gcol.data_ptr(), ws.data_ptr(), ws_bytes, _lib.stream_ptr()))
    torch.cuda.synchronize()
    return out.cpu(), gcol, gdep, galp


def _loss_twin(pred, gt, depth, gtd, alpha, boxes, w, dtype):
    """Values {out index: value} and (dL/dpred, dL/ddepth, dL/dalpha) of the loss stage's objective."""
    p, d, a = _leaves(dtype, CUDA, pred, depth, alpha)
    g, gd = gt.to(dtype), gtd.to(dtype)
    photo, l1, s = photometric(p, g, w["w_l1"], w["w_dssim"])
    vals = {0: photo, 1: l1, 2: s}
    total = photo
    if w["w_pearson"]:
        vals[3] = pearson(d, gd)
        total = total + w["w_pearson"] * vals[3]
    if w["w_alpha"]:
        vals[4] = alpha_term(a, w["w_alpha"])
        total = total + vals[4]
    if boxes and w["w_local"]:
        vals[5] = pearson_boxes(d, gd, boxes).mean()
        total = total + w["w_local"] * vals[5]
    grads = torch.autograd.grad(total, [p, d, a], allow_unused=True)
    grads = [torch.zeros_like(x) if gr is None else gr for gr, x in zip(grads, (p, d, a))]
    return {k: v.item() for k, v in vals.items()}, [gr.detach() for gr in grads]


def _loss_inputs(H, W, s, n_boxes, seed):
    """Images with a black background (pred = gt = 0), exact ties, saturated 0 / 1; depth up to ~100 with an all-zero
    box and a nearly constant box; boxes flush with the last row / column, three over one pixel, on and off the 32 grid."""
    g = torch.Generator().manual_seed(seed)
    a = torch.rand(3, H, W, generator=g)
    b = (a + 0.15 * torch.randn(3, H, W, generator=g)).clamp(0, 1)          # clamp: exact 0 and 1 in gt
    a[:, : H // 5, W // 2:] = 1.0                                          # saturated prediction
    a[:, H // 2:, : W // 3] = 0.0                                          # black background ...
    b[:, H // 2:, : W // 3] = 0.0                                          # ... on both sides
    tie = torch.rand(3, H, W, generator=g) < 0.1
    b[tie] = a[tie]
    d1 = torch.rand(1, H, W, generator=g) * 5 + torch.linspace(0, 95, W).reshape(1, 1, W)
    d2 = d1 * 0.7 + 0.5 * torch.rand(1, H, W, generator=g)
    zr, zc = (H - s) // 3, (W - s) // 3
    cr, cc = 2 * (H - s) // 3, 2 * (W - s) // 3
    d1[:, zr:zr + s, zc:zc + s] = 0.0                                      # rendered depth over empty space
    d1[:, cr:cr + s, cc:cc + s] = 5.0 + 1e-3 * torch.rand(1, s, s, generator=g)
    al = torch.rand(1, H, W, generator=g)
    r3, c3 = (H - s) // 2, (W - s) // 2
    r3, c3 = min(r3, H - s - s // 2), min(c3, W - s - s // 2)
    boxes = [(zr, zc), (cr, cc), (H - s, W - s), (r3, c3), (r3 + s // 4, c3 + s // 3), (r3 + s // 2, c3 + s // 2),
             (H - s, 0), (0, W - s), (0, 0), (min(32, H - s), min(64, W - s))]
    while len(boxes) < n_boxes:
        boxes.append((int(torch.randint(0, H - s + 1, (1,), generator=g)), int(torch.randint(0, W - s + 1, (1,), generator=g))))
    boxes = [(r, c, s, s) for r, c in boxes[:n_boxes]]
    return a, b, d1, d2, al, boxes, [(zr, zc, s, s), (cr, cc, s, s)]


def _depth_regions(H, W, special, device):
    """[(name, mask)]: the all-zero box and the nearly constant box (their ~1/eps and ~1/std(p) gradients would set
    max|b| for the whole map) each on its own, then the rest of the map; every pixel in exactly one region."""
    rest = torch.ones(1, H, W, dtype=torch.bool, device=device)
    out = []
    for name, (r, c, h, w) in zip(("zero box", "flat box"), special):
        m = torch.zeros_like(rest)
        m[:, r:r + h, c:c + w] = True
        m &= rest
        rest &= ~m
        out.append((name, m))
    return out + [("rest", rest)]


def _check_loss_stage(H, W, s, n_boxes, seed, w):
    a, b, d1, d2, al, boxes, special = _loss_inputs(H, W, s, n_boxes, seed)
    dev = [t.to(CUDA) for t in (a, b, d1, d2, al)]
    out, gcol, gdep, galp = _loss_stage(*dev, boxes, w)
    v64, g64 = _loss_twin(*dev, boxes, w, torch.float64)
    v32, g32 = _loss_twin(*dev, boxes, w, torch.float32)
    tag = f"{H}x{W} {n_boxes} boxes"
    for k in range(6):
        if k in v64:
            _value(f"{tag} out[{k}]", out[k], v64[k])
        else:
            assert out[k].item() == -1.0, f"{tag}: out[{k}] of a disabled term was written"
    _bar("rdg_losses dL/dpred", tag, gcol, g32[0], g64[0])
    if w["w_pearson"] or (boxes and w["w_local"]):
        for name, m in _depth_regions(H, W, special if boxes and w["w_local"] else [], CUDA):
            _bar("rdg_losses dL/ddepth", f"{tag} {name}", gdep, g32[1], g64[1], m)
    else:
        assert (gdep == 7.0).all()
    if w["w_alpha"]:
        want = torch.tensor(-w["w_alpha"], dtype=torch.float32).double() / (H * W)
        assert (galp == want.float().item()).all(), "dL/dalpha is not float32(-w_alpha / (H W))"
    else:
        assert (galp == 7.0).all()
    if w["w_l1"]:
        # at pred == gt the L1 term contributes nothing: the same call without L1 gives bit-identical gradients there
        _, gcol0, _, _ = _loss_stage(*dev, boxes, dict(w, w_l1=0.0))
        tie = dev[0] == dev[1]
        assert tie.any() and torch.equal(gcol[tie], gcol0[tie])
    return tag


def test_loss_workspace_keeps_the_local_boxes_aligned():
    """The LocalBox array behind the three derivative maps is read as float4: it must start on 16 bytes for every image
    size, including those whose C * H * W is not a multiple of 4 (33x70 faulted with a misaligned address before)."""
    from rodygs_b200 import _lib
    lib = _lib.load()
    for ch, H, W in ((3, 33, 70), (3, 97, 131), (1, 7, 9), (3, 1080, 1920), (3, 8, 8)):
        boxes_at = lib.rdg_l1_dssim_workspace_bytes(ch, H, W) - 256 * 64
        assert boxes_at % 16 == 0 and boxes_at >= 256 + 3 * ch * H * W * 4, (ch, H, W)
    assert lib.rdg_l1_dssim_workspace_bytes(3, 1080, 1920) == 256 + 3 * 3 * 1080 * 1920 * 4 + 256 * 64


LOSS_CASES = [(1080, 1920, 128, 60), (540, 960, 128, 14), (512, 512, 128, 8), (33, 70, 16, 33), (97, 131, 16, 33),
              (97, 131, 16, 256), (33, 70, 16, 256)]


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,s,n_boxes", LOSS_CASES)
def test_loss_stage_against_float64(H, W, s, n_boxes):
    _check_loss_stage(H, W, s, n_boxes, 100 + H, W4)


@pytest.mark.gpu
@pytest.mark.parametrize("off", ["w_pearson", "w_local", "w_alpha", "w_l1", "w_dssim", "depth"])
def test_loss_stage_terms_switched_off(off):
    w = dict(W4)
    for k in (("w_pearson", "w_local") if off == "depth" else (off,)):
        w[k] = 0.0
    _check_loss_stage(97, 131, 16, 40, 7, w)


# ---------------------------------------------------------------- rdg_pearson --

def _pearson_abi(pred, gt, boxes, weights, grad0):
    from rodygs_b200 import _lib
    lib = _lib.load()
    H, W = pred.shape[-2:]
    bx = torch.tensor(boxes, dtype=torch.int32, device=CUDA).contiguous()
    out = torch.full((len(boxes),), -1.0, device=CUDA)
    stats = torch.empty(len(boxes) * 8, dtype=torch.float64, device=CUDA)
    grad = grad0.clone()
    _lib.check(lib.rdg_pearson(pred.data_ptr(), gt.data_ptr(), H, W, bx.data_ptr(), _lib.ptr(weights), len(boxes), EPS,
                               out.data_ptr(), grad.data_ptr(), stats.data_ptr(), _lib.stream_ptr()))
    torch.cuda.synchronize()
    return out.cpu(), grad


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["whole_1080p", "rect60", "rect60_prefilled"])
def test_pearson_kernel_against_float64(case):
    H, W = 1080, 1920
    a, b, d1, d2, al, _, _ = _loss_inputs(H, W, 128, 0, 21)
    g = torch.Generator().manual_seed(22)
    pred, gt = d1.to(CUDA), d2.to(CUDA)
    if case == "whole_1080p":
        boxes, weights = [(0, 0, H, W)], None
    else:
        boxes = [(0, 0, 40, 300), (H - 200, W - 64, 200, 64), (H - 7, 0, 7, W), (0, W - 1, H, 1)]
        while len(boxes) < 60:
            h, w_ = int(torch.randint(2, 300, (1,), generator=g)), int(torch.randint(2, 300, (1,), generator=g))
            if h == w_:
                continue
            boxes.append((int(torch.randint(0, H - h + 1, (1,), generator=g)), int(torch.randint(0, W - w_ + 1, (1,), generator=g)), h, w_))
        weights = (torch.rand(60, generator=g) + 0.1).to(CUDA)
    grad0 = torch.zeros(1, H, W, device=CUDA)
    if case == "rect60_prefilled":
        grad0 = torch.randn(1, H, W, generator=g).to(CUDA) * 1e-6
    out, grad = _pearson_abi(pred, gt, boxes, weights, grad0)
    refs = {}
    for dtype in (torch.float32, torch.float64):
        (p,) = _leaves(dtype, CUDA, pred)
        per_box = pearson_boxes(p, gt.to(dtype), boxes)
        wts = torch.ones(len(boxes), dtype=dtype, device=CUDA) if weights is None else weights.to(dtype)
        (gr,) = torch.autograd.grad((per_box * wts).sum(), p)
        refs[dtype] = (per_box.detach().cpu(), grad0.to(dtype) + gr)
    for k in range(len(boxes)):
        _value(f"{case} box {k}", out[k], refs[torch.float64][0][k])
    _bar("rdg_pearson", case, grad, refs[torch.float32][1], refs[torch.float64][1])


# ================================================================ part 4: motion regularisers (GPU) ==

def _coeff_rows(n, seed):
    g = torch.Generator().manual_seed(seed)
    c = torch.randn(n, 16, generator=g) * 0.2
    v = torch.rand(n, 1, generator=g) + 0.5
    c[1::997, 3], c[1::997, 11] = v[1::997, 0], -v[1::997, 0]              # c and -c: two-way tie
    for k in (0, 4, 7, 15):                                                # four-way ties, mixed signs
        c[2::991, k] = v[2::991, 0] * (1 if k % 2 else -1)
    c[::1000] = 0.0                                                        # all-zero rows
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("accumulate", [False, True])
def test_coefficient_regularisers_against_float64(accumulate):
    from rodygs_b200 import motion_reg as mr
    n, wl, ws = 1_000_000, 0.01, 0.002
    c = _coeff_rows(n, 31).to(CUDA)
    refs = {}
    for dtype in (torch.float32, torch.float64):
        (x,) = _leaves(dtype, CUDA, c)
        l1, sp = motion_l1(x), motion_sparsity(x)
        (gr,) = torch.autograd.grad(wl * l1 + ws * sp, x)
        refs[dtype] = (l1.item(), sp.item(), gr)
    d0 = torch.randn(n, 16, device=CUDA) * refs[torch.float64][2].abs().max().float() if accumulate else \
        torch.full((n, 16), float("nan"), device=CUDA)
    d = d0.clone()
    parts = mr.motion_coeff_reg_(c, wl, ws, d, accumulate=accumulate).cpu()
    _value("mean|c|", parts[0], refs[torch.float64][0])
    _value("sparsity", parts[1], refs[torch.float64][1])
    got = d.double() - d0.double() if accumulate else d
    _bar("rdg_motion_coeff_reg", f"1M x 16 accumulate={accumulate}", got, refs[torch.float32][2], refs[torch.float64][2])
    zero = (c == 0).all(1)
    assert zero.sum() == 1000 and torch.equal(d[zero], d0[zero] if accumulate else torch.zeros_like(d[zero]))
    # ties: the max term goes to the first index, the others keep the plain |c| gradient
    g64 = refs[torch.float64][2]
    assert torch.equal(got[1::997, 11].sign(), g64[1::997, 11].sign().to(got.dtype))


@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 12, 100])
@pytest.mark.parametrize("mode", ["cum_exponential", "vanilla"])
@pytest.mark.parametrize("td,rd", [(0, 0), (0, -1), (-1, 0)])
def test_basis_regulariser_against_float64(T, mode, td, rd):
    from rodygs_b200 import motion_reg as mr
    g = torch.Generator().manual_seed(40 + T)
    tb = _basis_table(T, g).to(CUDA)
    reg = _reg(mode).to(CUDA)
    refs = {}
    for dtype in (torch.float32, torch.float64):
        (x,) = _leaves(dtype, CUDA, tb)
        t, r, loss = motion_basis_reg(x, reg.to(dtype), td, rd)
        (gr,) = torch.autograd.grad(loss, x)
        refs[dtype] = (t.item(), r.item(), gr)
    # entries of a disabled term hold other gradients already: they must come back bit-identical
    off = torch.zeros(T, 16, 7, dtype=torch.bool, device=CUDA)
    if td < 0:
        off[..., :3] = True
    if rd < 0:
        off[..., 3:] = True
    # the written entries hold gradients of the same size: the kernel adds (d0 + 0.1 g), it does not overwrite
    scale = 0.1 * refs[torch.float64][2].abs().max().float().item()
    d = torch.randn(T, 16, 7, device=CUDA) * torch.where(off, 1.0, scale)
    d0 = d.clone()
    parts = mr.motion_basis_reg_(tb, reg, td, rd, d, grad_scale=0.1).cpu()
    _value("translation", parts[0], refs[torch.float64][0])
    _value("rotation", parts[1], refs[torch.float64][1])
    assert torch.equal(d[off], d0[off])
    tag = f"T {T} {mode} td {td} rd {rd}"
    _bar("rdg_motion_basis_reg", tag, d[~off], (d0 + 0.1 * refs[torch.float32][2])[~off],
         (d0.double() + 0.1 * refs[torch.float64][2])[~off])
    # and what was added, alone (d0 ~ 0.1 max|g|: the subtraction costs < 1e-8 max|g|, far below the floor)
    _bar("rdg_motion_basis_reg", tag + " added", (d.double() - d0.double())[~off], 0.1 * refs[torch.float32][2][~off],
         0.1 * refs[torch.float64][2][~off])


# ---------------------------------------------------------------- rigidity --

def _cloud(n, seed, dup_frac=0.0):
    g = torch.Generator().manual_seed(seed)
    centres = torch.randn(max(n // 400, 4), 3, generator=g) * 2
    canon = centres[torch.randint(0, centres.shape[0], (n,), generator=g)] + torch.randn(n, 3, generator=g) * 0.4
    coeff = torch.randn(n, 16, generator=g) * 0.2
    pred = torch.randn(n, 3, generator=g) * 0.02
    nd = int(n * dup_frac)
    if nd:
        src, dst = torch.randperm(n, generator=g)[: 2 * nd].view(2, nd)
        canon[dst], coeff[dst], pred[dst] = canon[src], coeff[src], pred[src]     # densification's clones
    return canon, coeff, pred


def _rigidity_abi(points, canon, coeff, table, fi, d2, nn, surface, distance, d_table):
    """rdg_rigidity on the neighbours (d2, nn) that knn_points gave; d_table is added to."""
    from rodygs_b200 import _lib
    lib = _lib.load()
    n, K = nn.shape
    a = _lib.RdgRigidity()
    a.n, a.K, a.eps, a.mode_surface, a.mode_distance = n, K, EPS, int(surface), int(distance)
    parts = torch.zeros(2, device=CUDA)
    d_points, d_canon, d_coeff = torch.empty_like(points), torch.empty_like(canon), torch.empty_like(coeff)
    fi32 = fi.to(CUDA, torch.int32).contiguous()
    a.points, a.nn_idx, a.nn_dist2, a.loss_parts, a.d_points = points.data_ptr(), nn.data_ptr(), d2.data_ptr(), \
        parts.data_ptr(), d_points.data_ptr()
    if distance:
        a.num_basis, a.n_frames = 16, fi32.numel()
        a.canon, a.coeff, a.table, a.frame_indices = canon.data_ptr(), coeff.data_ptr(), table.data_ptr(), fi32.data_ptr()
        a.d_canon, a.d_coeff, a.d_table = d_canon.data_ptr(), d_coeff.data_ptr(), d_table.data_ptr()
    nbytes = int(lib.rdg_rigidity_workspace_bytes(n, K, fi32.numel() if distance else 0))
    ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=CUDA)
    _lib.check(lib.rdg_rigidity(C.byref(a), ws.data_ptr(), nbytes, _lib.stream_ptr()))
    torch.cuda.synchronize()
    return parts.cpu(), d_points, d_canon, d_coeff


def _check_rigidity(n, K, Ts, surface, distance, seed, dup_frac=0.0, T=None):
    T = T or max(Ts + 2, 12)
    g = torch.Generator().manual_seed(seed)
    canon, coeff, pred = (t.to(CUDA) for t in _cloud(n, seed, dup_frac))
    points = canon + pred
    table = (torch.randn(T, 16, 7, generator=g) * 0.1).to(CUDA)
    fi = torch.randint(0, T - 1, (Ts,), generator=g)
    from rodygs_b200 import motion_reg as mr
    d2, nn = mr.knn_points(points, K)
    refs = {}
    for dtype in (torch.float32, torch.float64):
        lv = _leaves(dtype, CUDA, points, canon, coeff, table)
        s, d = rigidity(*lv, fi.to(CUDA), nn, surface, distance)
        grads = torch.autograd.grad(s + d, lv, allow_unused=True)
        refs[dtype] = (s.item(), d.item(), [torch.zeros_like(x) if gr is None else gr for gr, x in zip(grads, lv)])
        del lv, s, d, grads
    r32, r64 = refs[torch.float32], refs[torch.float64]
    # d_table holds other gradients already: entries rigidity does not touch must come back bit-identical, the frames it
    # touches get the gradient added to gradients of the same size
    touched = torch.zeros(T, 16, 7, dtype=torch.bool, device=CUDA)
    if distance:
        touched[fi.to(CUDA), :, :3] = True
    scale = max(r64[2][3].abs().max().item(), 1e-30)
    d_table = torch.randn(T, 16, 7, device=CUDA) * torch.where(touched, scale, 1.0)
    d_table0 = d_table.clone()
    parts, d_points, d_canon, d_coeff = _rigidity_abi(points, canon, coeff, table, fi, d2, nn, surface, distance, d_table)
    tag = f"n {n} K {K} Ts {Ts} surface {surface} distance {distance} dup {dup_frac}"
    if surface:
        _value(tag + " surface", parts[0], r64[0])
    if distance:
        _value(tag + " distance", parts[1], r64[1])
    _bar("rdg_rigidity d_points", tag, d_points, r32[2][0], r64[2][0])
    if distance:
        _bar("rdg_rigidity d_canon", tag, d_canon, r32[2][1], r64[2][1])
        _bar("rdg_rigidity d_coeff", tag, d_coeff, r32[2][2], r64[2][2])
        _bar("rdg_rigidity d_table", tag, d_table[touched], (d_table0 + r32[2][3])[touched],
             (d_table0.double() + r64[2][3])[touched])
        _bar("rdg_rigidity d_table", tag + " added", (d_table.double() - d_table0.double())[touched], r32[2][3][touched],
             r64[2][3][touched])
    assert torch.equal(d_table[~touched], d_table0[~touched]), "rdg_rigidity wrote d_table entries it does not own"


RIGID_CASES = [(1, 3), (3, 1), (3, 8), (8, 1), (8, 3), (8, 25), (8, 275), (16, 8), (16, 275), (1, 275)]


@pytest.mark.gpu
@pytest.mark.parametrize("K,Ts", RIGID_CASES)
@pytest.mark.parametrize("mode", ["both", "surface", "distance"])
def test_rigidity_against_float64(K, Ts, mode):
    _check_rigidity(6000, K, Ts, mode != "distance", mode != "surface", 50 + K * 7 + Ts)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 8, 16])
def test_rigidity_with_exact_duplicates(K):
    _check_rigidity(8000, K, 8, True, True, 60 + K, dup_frac=0.05)


@pytest.mark.gpu
def test_rigidity_at_production_sample_size():
    _check_rigidity(250_000, 8, 25, True, True, 70, dup_frac=0.05, T=100)


# ---------------------------------------------------------------- sample gather / scatter and the trainer --

@pytest.mark.gpu
@pytest.mark.parametrize("nd,T,w_rig", [(200_000, 100, 0.5), (200_000, 100, 1.0), (3000, 300, 1.0)])
def test_trainer_motion_losses_against_float64(nd, T, w_rig):
    """SplatTrainStep.motion_losses_backward (coefficient and basis regularisers, rigidity on the sample deformed by
    rdg_rigidity_sample, scattered back by rdg_rigidity_sample_bwd) against the float64 composition; w_rigidity 1.0 takes
    the branch where rigidity adds into the flat table gradient directly, T = 300 the sample backward's shared-memory
    path above 48 KB."""
    from rodygs_b200 import _lib, motion_reg as mr, synthetic, trainer
    lib = _lib.load()
    H, W = 64, 96
    sc = synthetic.make_scene(2 * nd, H, W, T, seed=9, radius_px=4.0)
    sc["spatial_lr_scale"] = lr = 1.7
    step = trainer.SplatTrainStep(sc, H, W)
    assert step.nd == nd
    g = torch.Generator().manual_seed(10)
    basis_t = (torch.randn(16, 7, generator=g) * 0.05).to(CUDA)
    indice = torch.randperm(nd, generator=g)[: nd // 2]
    fi = torch.randint(0, T - 1, (T // 4,), generator=g)
    w = dict(w_motion_l1=0.01, w_sparsity=0.002, w_basis=0.1, w_rigidity=w_rig)
    step.grads.fill_(0.0)
    parts = step.motion_losses_backward(5, basis_t, indice=indice, frame_indices=fi, **w).cpu()
    got = [step.g("dynamic.xyz").view(nd, 3), step.g("motion_coeff").view(nd, 16), step.g("table").view(T, 16, 7),
           step.g("basis_t").view(16, 7)]
    # the kernel's neighbours: the same deterministic sample kernel on the same inputs, then the exact KNN
    idx = indice.to(CUDA, torch.int32)
    n = idx.numel()
    xyz, coeff, table = step.p("dynamic.xyz").view(nd, 3), step.p("motion_coeff").view(nd, 16), step.p("table").view(T, 16, 7)
    pts, canon, cs = torch.empty(n, 3, device=CUDA), torch.empty(n, 3, device=CUDA), torch.empty(n, 16, device=CUDA)
    _lib.check(lib.rdg_rigidity_sample(n, 16, idx.data_ptr(), xyz.data_ptr(), coeff.data_ptr(), step.time_ind.data_ptr(),
                                       basis_t.data_ptr(), table.data_ptr(), lr, pts.data_ptr(), canon.data_ptr(),
                                       cs.data_ptr(), _lib.stream_ptr()))
    _, nn = mr.knn_points(pts, 8)
    ti = step.time_ind
    reg = _reg("cum_exponential").to(CUDA)
    refs = {}
    for dtype in (torch.float32, torch.float64):
        x, c, tb, tbs, bt = _leaves(dtype, CUDA, xyz, coeff, table, table, basis_t)
        p_s = sample_points(x, c, tbs, bt, ti, idx.long(), lr)
        assert helpers.rel_err(p_s.detach().float(), pts) < 1e-5
        s, dpres = rigidity(p_s, x[idx.long()], c[idx.long()], tb, fi.to(CUDA), nn)
        vals = (motion_l1(c), motion_sparsity(c), *motion_basis_reg(tb, reg.to(dtype))[:2], s, dpres)
        total = w["w_motion_l1"] * vals[0] + w["w_sparsity"] * vals[1] + w["w_basis"] * (vals[2] + vals[3]) + w_rig * (s + dpres)
        gx, gc, gt_, gts, gbt = torch.autograd.grad(total, [x, c, tb, tbs, bt])
        # d/dB(t) is minus the sum over frames of the table gradient of the sample term (the deformation sees B(t) - table)
        if dtype == torch.float64:
            assert helpers.elementwise_ok(gbt, -gts.sum(0), rtol=1e-9, floor=1e-12)[0]
        refs[dtype] = ([v.item() for v in vals], [gx, gc, gt_ + gts, gbt])
        del x, c, tb, tbs, bt, p_s, total
    tag = f"nd {nd} T {T} w_rig {w_rig}"
    for k in range(6):
        _value(f"{tag} motion_parts[{k}]", parts[k], refs[torch.float64][0][k])
    for name, a, r32, r64 in zip(("dynamic.xyz", "motion_coeff", "table", "basis_t"), got, refs[torch.float32][1],
                                 refs[torch.float64][1]):
        _bar(f"motion_losses_backward {name}", tag, a, r32, r64)

    # rdg_rigidity_sample_bwd alone, on zeroed outputs: B(t)'s gradient is minus the sum of the table's over the frames
    gu = torch.Generator().manual_seed(11)
    d_pts, d_can, d_cs = (torch.randn(*shape, generator=gu).to(CUDA) * 1e-3 for shape in ((n, 3), (n, 3), (n, 16)))
    outs = [torch.zeros(nd, 3, device=CUDA), torch.zeros(nd, 16, device=CUDA), torch.zeros(16, 7, device=CUDA),
            torch.zeros(T, 16, 7, device=CUDA)]
    _lib.check(lib.rdg_rigidity_sample_bwd(n, 16, T, idx.data_ptr(), coeff.data_ptr(), ti.data_ptr(), basis_t.data_ptr(),
                                           table.data_ptr(), lr, 0.5, d_pts.data_ptr(), d_can.data_ptr(), d_cs.data_ptr(),
                                           *[o.data_ptr() for o in outs], _lib.stream_ptr()))
    torch.cuda.synchronize()
    refs = {}
    for dtype in (torch.float32, torch.float64):
        x, c, tb, bt = _leaves(dtype, CUDA, xyz, coeff, table, basis_t)
        il = idx.long()
        p_s = sample_points(x, c, tb, bt, ti, il, lr)
        obj = 0.5 * ((p_s * d_pts.to(dtype)).sum() + (x[il] * d_can.to(dtype)).sum() + (c[il] * d_cs.to(dtype)).sum())
        refs[dtype] = torch.autograd.grad(obj, [x, c, bt, tb])
    for name, a, r32, r64 in zip(("d_xyz", "d_coeff", "d_basis_t", "d_table"), outs, refs[torch.float32], refs[torch.float64]):
        _bar("rdg_rigidity_sample_bwd", f"{tag} {name}", a, r32, r64)
    assert torch.equal(outs[3][..., 3:], torch.zeros_like(outs[3][..., 3:])) and torch.equal(outs[2][:, 3:], torch.zeros(16, 4, device=CUDA))
    ok, ratio = helpers.elementwise_ok(outs[2][:, :3], -outs[3].double().sum(0)[:, :3])
    assert ok, f"{tag}: d_basis_t != -sum over frames of d_table ({ratio:.3f} x the bar)"


# ================================================================ part 5: basis MLP backward (GPU) ==

def _relu_near_zero(net, emb, margin):
    """[rows] bool: a ReLU pre-activation of the row (timenet or head) within `margin` of zero."""
    h, near = emb, torch.zeros(emb.shape[0], dtype=torch.bool)
    for li in (0, 2, 4):
        z = net.timenet[li](h)
        near |= (z.abs() < margin).any(-1)
        h = torch.relu(z)
    w0 = torch.stack([hd.basis[0].weight for hd in net.basis_xyz])
    b0 = torch.stack([hd.basis[0].bias for hd in net.basis_xyz])
    z = torch.einsum("ri,koi->rko", h, w0) + b0
    return near | (z.abs() < margin).flatten(1).any(-1)


@pytest.mark.gpu
@pytest.mark.parametrize("width", [128, 256])
@pytest.mark.parametrize("act", ["gelu", "relu"])
@pytest.mark.parametrize("T", [100, 1])
def test_basis_mlp_backward_against_float64(width, act, T):
    from rodygs_b200 import deform
    torch.manual_seed(1000 + width + T)
    twin = deform.MotionBasisNetwork(width, 16, 26, False, activation=act)
    with torch.no_grad():
        for p in twin.parameters():
            p.copy_(torch.randn_like(p) * (1.5 / p.shape[1] ** 0.5 if p.dim() > 1 else 0.1))
        if act == "relu":                       # dead units: pre-activations below zero for every time
            twin.timenet[0].bias[: width // 8] = -50.0
            twin.timenet[2].bias[: width // 8] = -50.0
            twin.basis_xyz[3].basis[0].bias[:] = -50.0
    times = torch.cat((torch.tensor([0.4321]), torch.arange(T, dtype=torch.float32) / T))
    emb = twin.batch_embedding(times)                                            # [T + 1, 53]: B(t) row + the table
    d_basis = torch.randn(T + 1, 16, 7)
    if act == "relu":
        # a row whose float64 pre-activation lies within float32 rounding of 0 may take the other side of the ReLU in
        # the kernel: it gets a zero upstream gradient (the gradients are linear in it), so no such decision remains
        near = _relu_near_zero(copy.deepcopy(twin).double(), emb.double(), margin=1e-5)
        assert near.sum() <= max(1, (T + 1) // 20)
        d_basis[near] = 0.0
    net = deform.BasisMLP(width, 16, 26, False, activation=act)
    net.load_state_dict(twin.state_dict())
    net.forward_rows(emb=emb.cuda())
    net.backward_rows(d_basis.cuda())
    got = net.grad_state_dict()
    refs = {}
    for dtype in (torch.float32, torch.float64):
        tw = copy.deepcopy(twin).to(CUDA, dtype)
        (tw.bases(emb.to(CUDA, dtype)) * d_basis.to(CUDA, dtype)).sum().backward()
        refs[dtype] = {k: p.grad for k, p in tw.named_parameters()}
    if act == "relu":
        assert got["timenet.0.weight"][: width // 8].abs().max().item() == 0.0
    for k in refs[torch.float64]:
        _bar("rdg_basis_mlp_bwd", f"width {width} {act} T {T} {k}", got[k], refs[torch.float32][k], refs[torch.float64][k])
