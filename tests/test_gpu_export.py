"""Export as a 3D Gaussian Splatting PLY file on the device (rdg_export_3dgs, SplatTrainStep.export_3dgs, rodygs_b200.ply).

Yardsticks: static records are the raw parameters bit for bit and a file of them re-renders bit-identically; dynamic means
have the bits of rdg_track_attrs' positions (the preprocess's deformation); dynamic covariances are held to the float64
twin of test_export_ply.py on the float32 q' and scales the preprocess itself used, and to closed forms; a dynamic scene
exported at time t and re-imported as a static scene renders what the original renders at t."""
import os
import tempfile

import pytest
import torch

from test_export_ply import rot64, sigma_of, twin
from test_gpu_metrics import _same, _snapshot
from test_gpu_tracking import IMG_TOL, TABLE_SMEM_MAX, _cams, _camera_snapshot, _make_step, _track


def _trained_like(step, factor=6.0):
    """scale the quaternion columns of the motion table, so that |q'| = |normalize(q) + dq(t)| spans about [0.7, 1.3]"""
    if step.nd > 0:
        step.p("table")[..., 3:7] *= factor


def _params(step, tag):
    return {k: step.p(f"{tag}.{k}") for k in ("xyz", "scaling", "rotation", "opacity", "features_dc", "features_rest")}


def _sh_columns(p, n, degree):
    """f_dc and f_rest of the records: the transposed parameters, zero above the degree"""
    rest = p["features_rest"].clone()
    rest[:, (degree + 1) ** 2 - 1:, :] = 0.0
    return torch.cat([p["features_dc"].reshape(n, 3), rest.transpose(1, 2).reshape(n, 45)], 1)


def _activated(step, vm, pm, fx, fy, bt):
    """the float32 (xyz, s, q', opacity) [N, 11] the preprocess used at B(t) = bt"""
    from rodygs_b200 import engine
    engine.config.debug_activated = True
    try:
        scene, view = step._scene_view(vm, pm, fx, fy, bt)
        return engine.render_forward(scene, view, keep_for_backward=True)[4].geom["dbg_activated"]
    finally:
        engine.config.debug_activated = False


def _reimported(step, records):
    """write_ply -> read_ply -> import_models -> SplatTrainStep with the step's image size and SH degree"""
    from rodygs_b200 import checkpoint, ply, synthetic
    from rodygs_b200.trainer import SplatTrainStep
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "scene.ply")
        ply.write_ply(path, records)
        assert os.path.getsize(path) == len(ply.ply_header(records.shape[0])) + 248 * records.shape[0]
        scene = checkpoint.import_models(ply.read_ply(path))
    return SplatTrainStep(synthetic.to_device(scene, "cuda"), step.H, step.W, sh_degree=step.sh_degree, w_pearson=0.0)


@pytest.mark.gpu
def test_static_records_are_the_parameters_and_their_file_renders_bit_identically():
    """Static-only scene, SH degree 3: every record equals the raw parameters (torch.equal); export -> write_ply -> read_ply
    -> import_models -> SplatTrainStep renders colour, depth, alpha and radii bit-identical to the original."""
    step = _make_step(20_001, 97, 131, dynamic_fraction=0.0)
    rec = step.export_3dgs(None)
    assert rec.shape == (20_001, 62) and rec.dtype == torch.float32 and rec.is_cuda
    p, n = _params(step, "static"), step.ns
    want = torch.cat([p["xyz"], torch.zeros(n, 3, device="cuda"), _sh_columns(p, n, 3), p["opacity"], p["scaling"],
                      p["rotation"]], 1)
    assert torch.equal(rec.view(torch.int32), want.view(torch.int32))
    other = _reimported(step, rec)
    vms, pms, fx, fy, _ = _cams(step, 3, seed=4)
    for a, b in zip(step.render_views(vms, pms, fx, fy, None), other.render_views(vms, pms, fx, fy, None)):
        assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("dynamic_fraction,T", [(0.5, 6), (0.5, TABLE_SMEM_MAX), (0.5, TABLE_SMEM_MAX + 1), (1.0, 6),
                                                (1.0, TABLE_SMEM_MAX + 1), (0.0, 6)])
def test_means_are_the_tracked_positions(dynamic_fraction, T):
    """x y z of every record is torch.equal to engine.track's positions (rdg_track_attrs: the preprocess's deformation) at
    the same B(t): both table paths (T = 6, 137 | 138), N = 20 001 (not a multiple of the 256-Gaussian chunk), N_s = 0 and
    N_d = 0."""
    step = _make_step(20_001, 97, 131, T=T, dynamic_fraction=dynamic_fraction)
    _trained_like(step)
    vms, pms, fx, fy, bts = _cams(step, 3, seed=T)
    pos = _track(step, vms, pms, fx, fy, bts)[4]
    for m in range(3):
        rec = step.export_3dgs(bts[m] if step.nd > 0 else None)
        assert torch.equal(rec[:, 0:3], pos[m]), (m, (rec[:, 0:3] != pos[m]).any(1).sum().item())
        assert (rec[:, 3:6] == 0).all()


def _check_records(rec, act, ns):
    """dynamic records against the twin on the preprocess's float32 q' and s: relative Frobenius error <= 1e-5, unit rot
    with rot_0 >= 0, finite; returns |q'| of the dynamic rows"""
    qp, s = act[ns:, 6:10].cpu(), act[ns:, 3:6].cpu()
    sigma = twin(qp, s)[0]
    rot, scale = rec[ns:, 58:62].cpu(), rec[ns:, 55:58].cpu()
    assert torch.isfinite(rot).all() and torch.isfinite(scale).all()
    got = sigma_of(rot, scale)
    err = (got - sigma).flatten(1).norm(dim=1) / sigma.flatten(1).norm(dim=1)
    assert err.max() <= 1e-5, (err.max().item(), err.argmax().item())
    assert ((rot.double().norm(dim=1) - 1).abs() <= 1e-6).all() and (rot[:, 0] >= 0).all()
    return qp.double().norm(dim=1)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [6, TABLE_SMEM_MAX + 1])
def test_dynamic_covariance_is_the_rasterizers(T):
    """Trained-like dq (|q'| over about [0.7, 1.3]): R(rot) diag(exp(2 scale)) R(rot)^T rebuilt in float64 from the records
    equals the twin's Sigma of the float32 q', s the preprocess used (dbg_activated) within 1e-5 relative Frobenius."""
    step = _make_step(20_001, 97, 131, T=T, dynamic_fraction=0.5)
    _trained_like(step)
    vms, pms, fx, fy, bts = _cams(step, 2, seed=1)
    for m in range(2):
        act = _activated(step, vms[m], pms[m], fx, fy, bts[m])
        norms = _check_records(step.export_3dgs(bts[m]), act, step.ns)
        assert norms.min() < 0.8 and norms.max() > 1.2, (norms.min().item(), norms.max().item())


@pytest.mark.gpu
def test_dynamic_covariance_closed_forms():
    """dq set through the motion basis (B(t) rows 0-3 carry unit quaternion columns, the coefficients carry dq, the table
    and the motion of the means are zero): q' = lambda q^ for a quarter turn with lambda^2 = 1.1 and a half turn with
    lambda^2 = 0.5 (singular), against Sigma = R(q') S^2 R(q')^T in closed form; the means do not move."""
    import numpy as np
    step = _make_step(2_000, 97, 131, T=6, dynamic_fraction=1.0)
    nd, K = step.nd, step.num_basis
    g = torch.Generator(device="cuda").manual_seed(2)
    quarter = torch.tensor([np.cos(np.pi / 4), 0, 0, np.sin(np.pi / 4)], dtype=torch.float32, device="cuda")
    half = torch.tensor([0.0, 0, 0, 1.0], device="cuda")
    lam = torch.where(torch.arange(nd, device="cuda") % 2 == 0, torch.tensor(1.1, device="cuda").sqrt(),
                      torch.tensor(0.5, device="cuda").sqrt())
    qhat = torch.where((torch.arange(nd, device="cuda") % 2 == 0)[:, None], quarter, half)
    step.p("dynamic.rotation").copy_(qhat * (0.5 + torch.rand(nd, 1, device="cuda", generator=g)))   # any length
    coeff = torch.zeros(nd, K, device="cuda")
    coeff[:, 0:4] = (lam[:, None] - 1.0) * qhat
    step.p("motion_coeff").view(nd, K).copy_(coeff)
    step.p("table").zero_()
    bt = torch.zeros(K, 7, device="cuda")
    bt[0:4, 3:7] = torch.eye(4, device="cuda")
    rec = step.export_3dgs(bt)
    assert torch.equal(rec[:, 0:3], step.p("dynamic.xyz"))
    s = step.p("dynamic.scaling").exp().double().cpu()
    qp = (lam.double()[:, None] * qhat.double()).cpu()
    closed = rot64(qp) @ torch.diag_embed(s * s) @ rot64(qp).transpose(1, 2)
    got = sigma_of(rec[:, 58:62].cpu(), rec[:, 55:58].cpu())
    err = (got - closed).flatten(1).norm(dim=1) / closed.flatten(1).norm(dim=1)
    assert err.max() <= 1e-5, err.max().item()
    assert torch.isfinite(rec).all()
    naive = sigma_of(qp, s.log())                                   # what q' written as it is would draw
    nerr = (naive - closed).flatten(1).norm(dim=1) / closed.flatten(1).norm(dim=1)
    assert nerr[0::2].min() > 0.01
    # the singular ones (R(q') = diag(0, 0, 1) up to float32 rounding): two axes below 1e-4 of the third
    sc = rec[1::2, 55:58].sort(1).values
    assert (sc[:, 1] < sc[:, 2] + np.log(1e-4)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("sh_degree", [0, 3])
def test_dynamic_scene_at_time_t_reimported_renders_the_same(sh_degree):
    """Export at B(t), re-import the file as a static scene: render_views at the same cameras agrees with the original's
    render at B(t) - radii equal, colour, depth and alpha within 1e-4 max-abs - at 97x131."""
    step = _make_step(5_001, 97, 131, T=6, sh_degree=sh_degree, dynamic_fraction=0.5, seed=5)
    _trained_like(step)
    vms, pms, fx, fy, bts = _cams(step, 3, seed=6)
    for m in range(2):
        other = _reimported(step, step.export_3dgs(bts[m]))
        ref = step.render_views(vms, pms, fx, fy, bts[m:m + 1].expand(3, -1, -1).contiguous())
        got = other.render_views(vms, pms, fx, fy, None)
        assert torch.equal(got[3], ref[3]), (m, (got[3] != ref[3]).sum().item())
        for a, b in zip(got[:3], ref[:3]):
            assert (a - b).abs().max() <= IMG_TOL, (m, (a - b).abs().max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("sh_degree", [0, 1, 2, 3])
def test_sh_above_the_degree_is_zero(sh_degree):
    """f_dc and f_rest are the transposed parameters up to the step's SH degree and 0 above it, static and dynamic rows."""
    step = _make_step(3_001, 97, 131, T=6, sh_degree=sh_degree)
    _, _, _, _, bts = _cams(step, 1)
    rec = step.export_3dgs(bts[0])
    for tag, rows in (("static", rec[:step.ns]), ("dynamic", rec[step.ns:])):
        p = _params(step, tag)
        assert torch.equal(rows[:, 6:54], _sh_columns(p, rows.shape[0], sh_degree)), tag
        assert torch.equal(rows[:, 54:55], p["opacity"])
    k = (sh_degree + 1) ** 2 - 1
    for c in range(3):
        assert (rec[:, 9 + 15 * c + k:9 + 15 * (c + 1)] == 0).all()


@pytest.mark.gpu
def test_export_leaves_the_training_state_alone():
    """After forward_backward (+ exchange_grads(defer_sh=True)), densification statistics, both optimisers and a camera table:
    every piece of training state is bit-identical after export_3dgs, the duplicate capacity is untouched, and two calls
    return the same bits; the deferred factors are still consumed by the next optimizer step."""
    from rodygs_b200 import engine
    from rodygs_b200.optim import CameraLRs, GaussianLRs
    step = _make_step(20_000, 176, 208)
    step.attach_optimizer("static", GaussianLRs())
    step.attach_optimizer("dynamic", GaussianLRs(scaling_lr=0.001, motion_coeff_lr=1.6e-4))
    step.enable_densification("static")
    step.enable_densification("dynamic")
    step.enable_factored_exchange(views_per_rank=1, world_size=1)
    vms, pms, fx, fy, bts = _cams(step, 3)
    step.enable_camera_learning(vms[:2].contiguous(), CameraLRs(1e-4, 1e-4))
    gt = torch.rand(3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    for it in (1, 2):
        step.forward_backward(vms[0], pms[0], fx, fy, bts[0], gt, None, dcolor_slot=0)
        step.exchange_grads(vms[:1].contiguous(), bts[:1].contiguous(), defer_sh=True)
        if it == 1:
            for tag in ("static", "dynamic"):
                step.add_densification_stats(tag)
                step.optimizer_step(tag, it)
    torch.cuda.synchronize()
    before, cams = _snapshot(step), _camera_snapshot(step)
    cap = {k: dict(v) for k, v in engine._capacity.items()}
    first, second = step.export_3dgs(bts[1]), step.export_3dgs(bts[1])
    torch.cuda.synchronize()
    after = _snapshot(step)
    assert torch.equal(first.view(torch.int32), second.view(torch.int32))
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
    """Under config.sync_free a pending duplicate count (claimed truncated here) is neither read nor cleared by export_3dgs:
    the next forward_backward raises the overflow that belongs to it."""
    from rodygs_b200 import engine
    step = _make_step(20_000, 176, 208)
    vms, pms, fx, fy, bts = _cams(step, 2)
    ref = step.export_3dgs(bts[0])
    gt = torch.rand(3, 176, 208, device="cuda", generator=torch.Generator(device="cuda").manual_seed(6))
    saved = engine.config.sync_free
    engine.config.sync_free = True
    try:
        step.forward_backward(vms[0], pms[0], fx, fy, bts[0], gt, None)
        st = engine._cap_state(step.params.device, step.ns + step.nd)
        host, ev, _ = st["pending"]
        st["pending"] = pending = (host, ev, 1)
        cap = st["cap"]
        got = step.export_3dgs(bts[0])
        assert st["pending"] is pending and st["cap"] == cap
        assert torch.equal(got.view(torch.int32), ref.view(torch.int32))
        with pytest.raises(RuntimeError, match="truncated"):
            step.forward_backward(vms[0], pms[0], fx, fy, bts[0], gt, None)
    finally:
        engine.config.sync_free = saved
        engine._cap_state(step.params.device, step.ns + step.nd)["pending"] = None
