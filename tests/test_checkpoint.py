"""Checkpoints of the flat-buffer trainer: SplatTrainStep.state_dict / load_state_dict / from_state_dict / save / load, and
the reference-named export / import of its models (rodygs_b200.checkpoint).

CPU tests run the host logic on a step whose buffers live on the CPU (built without its CUDA-only constructor); the GPU
tests resume a real training run and compare it with the uninterrupted one."""
import hashlib
import math
import types

import pytest
import torch

from rodygs_b200 import checkpoint as ck
from rodygs_b200 import optim as ro
from rodygs_b200 import synthetic
from rodygs_b200.trainer import PARAM_ORDER, SplatTrainStep


# ---------------------------------------------------------------------------------------- CPU

def _cpu_step(n=300, T=5, K=16, H=64, W=96, seed=0):
    """A SplatTrainStep whose buffers live on the CPU: the attributes __init__ sets, minus the CUDA-only ones."""
    step = SplatTrainStep.__new__(SplatTrainStep)
    step.dev = torch.device("cpu")
    step.H, step.W, step.sh_degree = H, W, 3
    step.w, step.w_local, step.box_p, step.n_local = (0.8, 0.2, 0.05, 0.0), 0.15, 32, 3
    step.pg, step.optim, step._skip_step, step.stats, step._deferred = None, {}, set(), {}, None
    step._load_scene(synthetic.make_scene(n, H, W, T, seed=seed, num_basis=K))
    return step


def _fake_mlp(K=16, T=5):
    sd = {"timenet.0.weight": torch.randn(8, 53), "basis_xyz.0.basis.0.bias": torch.randn(4)}
    mlp = types.SimpleNamespace(num_basis=K, state_dict=lambda: {k: v.clone() for k, v in sd.items()},
                                init_args={"netwidth": 128, "num_basis": K, "t_emb_multires": 26, "t_log_sampling": False,
                                           "activation": "gelu", "out_dim": 7})
    return mlp, sd


def _attach_fake_mlp(step, K=16):
    mlp, sd = _fake_mlp(K, step.T)
    step.mlp = mlp
    step._mlp_times = torch.cat((torch.zeros(1), torch.arange(step.T, dtype=torch.float32) / step.T))
    step._mlp_lr, step._mlp_steps = 1e-3, 4
    step._mlp_moments = (torch.randn(10), torch.rand(10))
    return sd


def _populate(step):
    """Optimisers with moments and steps, statistics, an armed skip: every field a resume must carry."""
    g = torch.Generator().manual_seed(1)
    step.attach_optimizer("static", ro.GaussianLRs())
    step.attach_optimizer("dynamic", ro.GaussianLRs(scaling_lr=0.001, motion_coeff_lr=1.6e-4))
    for tag, opt in step.optim.items():
        for group in opt.ranges:
            m, v = opt.moments(group)
            m.copy_(torch.randn(m.shape, generator=g))
            v.copy_(torch.rand(v.shape, generator=g))
        opt.steps = 7 if tag == "static" else 6
        st = step.enable_densification(tag)
        st.grad_accum.copy_(torch.rand(st.n, generator=g))
        st.denom.copy_(torch.randint(0, 5, (st.n,), generator=g).float())
        st.max_radii2D.copy_(torch.rand(st.n, generator=g) * 9)
    step._skip_step.add("dynamic")


@pytest.fixture
def cpu_rng(monkeypatch):
    """The CUDA generator state stands in as the CPU generator's on a machine without a GPU."""
    monkeypatch.setattr(torch.cuda, "get_rng_state", lambda device=None: torch.get_rng_state())
    monkeypatch.setattr(torch.cuda, "set_rng_state", lambda state, device=None: torch.set_rng_state(state))


def _assert_same_state(a, b):
    assert (a.ns, a.nd, a.num_basis, a.T, a.H, a.W, a.sh_degree) == (b.ns, b.nd, b.num_basis, b.T, b.H, b.W, b.sh_degree)
    assert a.w == b.w and (a.w_local, a.box_p, a.n_local) == (b.w_local, b.box_p, b.n_local)
    assert torch.equal(a.params, b.params) and torch.equal(a.time_ind, b.time_ind)
    assert a.spatial_lr_scale == b.spatial_lr_scale and a._skip_step == b._skip_step
    assert a.optim.keys() == b.optim.keys() and a.stats.keys() == b.stats.keys()
    for tag, o in a.optim.items():
        p = b.optim[tag]
        assert o.steps == p.steps and o.lrs == p.lrs and tuple(o.betas) == tuple(p.betas) and o.eps == p.eps, tag
        assert torch.equal(o.exp_avg, p.exp_avg) and torch.equal(o.exp_avg_sq, p.exp_avg_sq), tag
    for tag, s in a.stats.items():
        t = b.stats[tag]
        for f in ("grad_accum", "denom", "max_radii2D"):
            assert torch.equal(getattr(s, f), getattr(t, f)), (tag, f)


def test_state_dict_survives_weights_only_load(tmp_path, cpu_rng):
    step = _cpu_step()
    _populate(step)
    mlp_sd = _attach_fake_mlp(step)
    sd = step.state_dict()
    assert set(sd["params"]) == set(step.layout) and "params" not in sd["optim"]["static"]
    assert sd["optim"]["dynamic"]["exp_avg"]["motion_coeff"].shape == (step.nd, 1, 16)
    assert sd["optim"]["static"]["exp_avg"]["f_rest"].shape == (step.ns, 15, 3)
    assert "motion_coeff_lr" not in sd["optim"]["static"]["lrs"]            # None fields are left out
    assert sd["skip_step"] == ["dynamic"] and sd["mlp"]["steps"] == 4
    torch.save(sd, tmp_path / "ck.pt")
    back = torch.load(tmp_path / "ck.pt", weights_only=True)

    def same(x, y):
        if torch.is_tensor(x):
            return torch.is_tensor(y) and x.dtype == y.dtype and torch.equal(x, y)
        if isinstance(x, dict):
            return isinstance(y, dict) and x.keys() == y.keys() and all(same(x[k], y[k]) for k in x)
        if isinstance(x, list):
            return isinstance(y, list) and len(x) == len(y) and all(same(u, v) for u, v in zip(x, y))
        return type(x) is type(y) and x == y

    assert same(sd, back)
    assert all(torch.equal(back["mlp"]["state_dict"][k], v) for k, v in mlp_sd.items())


def test_load_state_dict_rebuilds_a_step_of_another_size(cpu_rng):
    """Densification changes N, so a resume loads into a step built for another count: the layout follows the state."""
    src = _cpu_step(n=300, seed=0)
    _populate(src)
    dst = _cpu_step(n=170, seed=4)
    dst.attach_optimizer("static", ro.GaussianLRs(feature_lr=0.5))       # replaced, not merged
    dst.sh_degree, dst.w, dst.w_local, dst.box_p, dst.n_local = 1, (1.0, 0.0, 0.0, 0.3), 0.0, 64, 0   # restored too
    dst.load_state_dict(src.state_dict())
    _assert_same_state(src, dst)
    assert torch.equal(dst.p("basis_t"), src.p("basis_t"))


def test_malformed_state_leaves_the_step_untouched(cpu_rng):
    """Every check runs before the step changes: a missing or misshapen entry raises and the step is as it was."""
    src = _cpu_step(n=300)
    _populate(src)
    sd = src.state_dict()
    dst = _cpu_step(n=170, seed=4)
    before = dst.params.clone()
    broken = [{**sd, "params": {k: v for k, v in sd["params"].items() if k != "table"}},
              {**sd, "optim": {"dynamic": {**sd["optim"]["dynamic"], "exp_avg": {}}}},
              {**sd, "ranks": [{**sd["ranks"][0], "stats": {"static": {**sd["ranks"][0]["stats"]["static"],
                                                                       "denom": torch.zeros(3)}}}]},
              {**sd, "time_ind": sd["time_ind"][:-1]}]
    for bad in broken:
        with pytest.raises(ValueError, match="load_state_dict: "):
            dst.load_state_dict(bad)
        assert dst.ns + dst.nd == 170 and torch.equal(dst.params, before) and not dst.optim and not dst.stats


def test_rank_entries_follow_the_loading_ranks(cpu_rng, monkeypatch):
    """Data parallel: each rank accumulates its own densification statistics between densifications.  A file saved by
    two ranks gives each of two ranks its own entry; one process gets the sums / maximum of both (what the next
    densify_and_prune would have all-reduced); on more ranks rank 0 carries the sums and the others start from zero."""
    src = _cpu_step()
    _populate(src)
    sd = src.state_dict()
    r0 = sd["ranks"][0]
    r1 = {"stats": {tag: {f: t * 3 + 1 for f, t in s.items()} for tag, s in r0["stats"].items()},
          "cuda_rng_state": torch.Generator().manual_seed(7).get_state()}
    sd["ranks"] = [r0, r1]
    for (rank, world), want in (((1, 2), r1["stats"]), ((0, 2), r0["stats"])):
        monkeypatch.setattr(SplatTrainStep, "_dp_rank_world", lambda self, rw=(rank, world): rw)
        dst = _cpu_step(n=170, seed=4).load_state_dict(sd)
        for tag, s in want.items():
            for f, t in s.items():
                assert torch.equal(getattr(dst.stats[tag], f), t), (rank, tag, f)
    for rank, world in ((0, 1), (0, 3), (2, 3)):
        monkeypatch.setattr(SplatTrainStep, "_dp_rank_world", lambda self, rw=(rank, world): rw)
        dst = _cpu_step(n=170, seed=4).load_state_dict(sd)
        for tag, s in r0["stats"].items():
            t = r1["stats"][tag]
            st = dst.stats[tag]
            assert torch.equal(st.max_radii2D, torch.maximum(s["max_radii2D"], t["max_radii2D"])), (rank, world, tag)
            for f in ("grad_accum", "denom"):
                want = s[f] + t[f] if rank == 0 else torch.zeros_like(s[f])
                assert torch.equal(getattr(st, f), want), (rank, world, tag, f)


def test_refusals_name_the_field(cpu_rng):
    src = _cpu_step()
    sd = src.state_dict()
    for field, kw in (("H", {"H": 80}), ("W", {"W": 112})):
        with pytest.raises(ValueError, match=rf"load_state_dict: {field} is "):
            _cpu_step(**kw).load_state_dict(sd)
    other = _cpu_step(K=8)
    _attach_fake_mlp(other, K=8)
    with pytest.raises(ValueError, match="num_basis is 16 in the state dict but the attached basis MLP has 8"):
        other.load_state_dict(sd)
    shorter = _cpu_step(T=4)
    _attach_fake_mlp(shorter)
    with pytest.raises(ValueError, match="T is 5 in the state dict but the attached basis MLP has 4"):
        shorter.load_state_dict(sd)
    with pytest.raises(ValueError, match="not a rodygs_b200.SplatTrainStep"):
        src.load_state_dict({**sd, "version": 99})
    # an attached network whose next basis_forward would overwrite the saved table
    with_mlp = _cpu_step()
    _attach_fake_mlp(with_mlp)
    before = with_mlp.params.clone()
    with pytest.raises(ValueError, match="no basis MLP but one is attached"):
        with_mlp.load_state_dict(sd)
    assert torch.equal(with_mlp.params, before)
    # exchange_grads(defer_sh=True) holds dL/dSH as factors the next optimizer_step consumes: not state, so no save
    src._deferred = {"pending": {"static"}}
    with pytest.raises(RuntimeError, match=r"pending; call optimizer_step"):
        src.state_dict()
    src._deferred["pending"].clear()             # both models stepped: nothing pending any more
    src.state_dict()


def test_export_import_names_and_shapes():
    step = _cpu_step(n=300, T=5)
    _attach_fake_mlp(step)
    d = ck.export_models(step)
    for tag, n in (("static", step.ns), ("dynamic", step.nd)):
        shapes = {"_xyz": (n, 3), "_scaling": (n, 3), "_rotation": (n, 4), "_opacity": (n, 1), "_features_dc": (n, 1, 3),
                  "_features_rest": (n, 15, 3)}
        for k, shp in shapes.items():
            assert tuple(d[tag][k].shape) == shp, (tag, k)
            assert torch.equal(d[tag][k], step.p(f"{tag}.{k[1:]}")), (tag, k)
    dyn = d["dynamic"]
    assert set(d["static"]) == {f"_{k}" for k in PARAM_ORDER}
    assert tuple(dyn["_motion_coeff"].shape) == (step.nd, 1, 16)
    assert dyn["gaussian_to_time_ind"].dtype == torch.int64 and torch.equal(dyn["gaussian_to_time_ind"], step.time_ind.long())
    assert torch.equal(dyn["gaussian_to_time"], step.time_ind.float() / step.T)
    assert set(dyn["_deform_network"]) == {"timenet.0.weight", "basis_xyz.0.basis.0.bias"}
    # the export is a copy: the next densification replaces the flat buffers
    step.params.zero_()
    assert float(d["static"]["_xyz"].abs().sum()) > 0
    scene = ck.import_models(d)
    assert scene["time_ind"].dtype == torch.int32 and scene["spatial_lr_scale"] == step.spatial_lr_scale
    for tag in ("static", "dynamic"):
        for k in PARAM_ORDER:
            assert torch.equal(scene[tag][k], d[tag][f"_{k}"]), (tag, k)
    assert torch.equal(scene["motion_coeff"], dyn["_motion_coeff"]) and torch.equal(scene["table"], d["motion"]["table"])
    # a model without the step's extras (what the reference trains) needs the table from the caller
    ref = {"static": d["static"], "dynamic": dyn}
    with pytest.raises(ValueError, match="no motion table"):
        ck.import_models(ref)
    scene = ck.import_models(ref, table=d["motion"]["table"], spatial_lr_scale=2.5)
    assert scene["spatial_lr_scale"] == 2.5 and "basis_t" not in scene
    bad = {"static": d["static"], "dynamic": {**dyn, "gaussian_to_time_ind": dyn["gaussian_to_time_ind"] + step.T}}
    with pytest.raises(ValueError, match=r"must lie in \[0, 5\)"):
        ck.import_models(bad, table=d["motion"]["table"])
    with pytest.raises(ValueError, match="static._opacity has shape"):
        ck.import_models({"static": {**d["static"], "_opacity": d["static"]["_opacity"].view(-1)}, "dynamic": dyn},
                         table=d["motion"]["table"])


# ---------------------------------------------------------------------------------------- GPU

def _make_step(N=20_000, H=160, W=224, T=6, seed=3, box_p=32):
    """box_p = 32 so that 160 x 224 holds local Pearson boxes: int(0.5 * 5 * 7) = 17 random boxes per step."""
    scene = synthetic.to_device(synthetic.make_scene(N, H, W, T, seed=seed), "cuda")
    step = SplatTrainStep(scene, H, W, sh_degree=3, w_pearson=0.05, box_p=box_p)
    cam = synthetic.make_camera(1, 8, H, W, T)
    vm = cam.world_view_transform.t().contiguous().cuda()
    pm = cam.projection_matrix.t().contiguous().cuda()
    gen = torch.Generator(device="cuda").manual_seed(5)
    gt = torch.rand(3, H, W, device="cuda", generator=gen) * 0.5 + 0.25
    gt_depth = 2.0 + 4.0 * torch.rand(1, H, W, device="cuda", generator=gen)
    return step, cam, vm, pm, gt, gt_depth


def _cams(H=160, W=224, T=6):
    out = []
    for v in range(8):
        c = synthetic.make_camera(v, 8, H, W, T)
        out.append((c.world_view_transform.t().contiguous().cuda(), c.projection_matrix.t().contiguous().cuda(), c.tanfovx,
                    c.tanfovy, c.time))
    return out


def _setup_training(step, T=6):
    from rodygs_b200.deform import BasisMLP
    step.attach_optimizer("static", ro.GaussianLRs(feature_lr=0.02))
    step.attach_optimizer("dynamic", ro.GaussianLRs(feature_lr=0.02, scaling_lr=0.001, motion_coeff_lr=1.6e-4))
    step.enable_densification("static")
    step.enable_densification("dynamic")
    torch.manual_seed(11)                       # BasisMLP draws its initial weights from the CPU generator
    step.attach_basis_mlp(BasisMLP(128, 16, 26, False), torch.arange(T, dtype=torch.float32) / T, lr=1e-3)


def _iteration(step, it, tag, cams, gt, gt_depth, parts, after_densify=None):
    """One half-iteration of the alternating loop: render + losses + backward, statistics, the MLP on dynamic turns,
    densify_and_prune of the dynamic model at iteration 6, then the model's optimizer step."""
    vm, pm, tx, ty, t = cams[(2 * it + (tag == "dynamic")) % len(cams)]
    bt = step.basis_forward(t)
    parts.append(step.forward_backward(vm, pm, tx, ty, bt, gt, gt_depth).clone())
    step.add_densification_stats(tag)
    if tag == "dynamic":
        step.basis_backward()
        step.basis_optimizer_step()
    if it == 6 and tag == "dynamic":
        st = step.stats["dynamic"]
        thr = float(torch.quantile((st.grad_accum / st.denom.clamp(min=1))[st.denom > 0], 0.7))
        step.densify_and_prune("dynamic", thr, 0.005, 4.0, None, generator=torch.Generator(device="cuda").manual_seed(0))
        if after_densify is not None:
            after_densify(step)
    step.optimizer_step(tag, it)


def _train(step, its, cams, gt, gt_depth, parts, after_densify=None):
    for it in its:
        for tag in ("static", "dynamic"):
            _iteration(step, it, tag, cams, gt, gt_depth, parts, after_densify)


def _assert_bit_equal(a, b, pa, pb):
    _assert_same_state(a, b)
    assert torch.equal(a.mlp.params, b.mlp.params) and a._mlp_steps == b._mlp_steps
    assert all(torch.equal(x, y) for x, y in zip(a._mlp_moments, b._mlp_moments))
    assert len(pa) == len(pb)
    for k, (x, y) in enumerate(zip(pa, pb)):
        assert torch.equal(x, y), (k, x.tolist(), y.tolist())


@pytest.mark.gpu
def test_resumed_run_matches_the_uninterrupted_run_bit_for_bit(tmp_path):
    """Deterministic backward (rdg_blend_bwd_deterministic + the one-CTA per-Gaussian backward); the local Pearson boxes
    are drawn from the CUDA generator every step.  Run A trains 12 iterations; run B saves right after the densification
    of iteration 6, before the skipped optimizer step, and is resumed twice: from_state_dict, and load into a step built
    on a scene of another size.  Parameters, Adam state, MLP and its Adam state, statistics and every iteration's loss
    parts must equal run A's exactly; the second restore starts from other loss weights, SH degree and box size.

    Why equality and not a bound: the one order-dependent sum left in this mode is the loss stage's, which adds its
    per-block float64 partials with atomics (csrc/loss.cu).  Those sums reach the rest of the step only through float32
    casts in the one-thread finalize kernels - 6 loss parts and 4 + 4 x 17 Pearson / alpha coefficients per step; the
    per-pixel gradients are float32 arithmetic on those coefficients.  Reordering a float64 sum moves it by ~1e-16
    relative, which changes a float32 rounding with probability ~2 x 1e-16 / 2^-24 = 3e-9 per value, ~6e-6 for the 24
    steps here.  On an NVIDIA B200 (1000 W limit) the uninterrupted 12 iterations also gave the same parameters,
    moments, MLP, statistics and loss parts bit for bit in two separate processes."""
    from rodygs_b200 import engine
    saved = engine.config.deterministic
    engine.config.deterministic = True
    try:
        cams = _cams()
        run_a, _, _, _, gt, gt_depth = _make_step()
        assert run_a.local_box_origins is None and run_a.n_local == 17
        _setup_training(run_a)
        parts_a = []
        _train(run_a, range(1, 13), cams, gt, gt_depth, parts_a)
        assert run_a.optim["dynamic"].steps == 11 and run_a.optim["static"].steps == 12

        run_b, *_ = _make_step()
        _setup_training(run_b)
        parts_b = []
        path = tmp_path / "step.pt"

        def save(step):
            assert step._skip_step == {"dynamic"}
            step.save(path)

        _train(run_b, range(1, 7), cams, gt, gt_depth, parts_b, after_densify=save)
        assert run_b.nd != 10_000
        for k in range(len(parts_b)):
            assert torch.equal(parts_a[k], parts_b[k]), k
        del run_b

        def from_file():
            return SplatTrainStep.from_state_dict(torch.load(path, weights_only=True))

        def into_other_size():
            scene = synthetic.to_device(synthetic.make_scene(12_000, 160, 224, 6, seed=8), "cuda")
            other = SplatTrainStep(scene, 160, 224, sh_degree=1, w_l1=1.0, w_dssim=0.0, w_pearson=0.0, w_local=0.0, box_p=64)
            assert other.nd != torch.load(path, weights_only=True)["nd"] and other.n_local == 0
            return other.load(path)

        # each restore right before its own run: the load also restores the CUDA generator both runs draw boxes from
        for restore in (from_file, into_other_size):
            step = restore()
            # what the run was going to do next: iteration 6's dynamic optimizer step (the post-densification no-op)
            steps = step.optim["dynamic"].steps
            step.optimizer_step("dynamic", 6)
            assert step.optim["dynamic"].steps == steps and not step._skip_step
            parts = list(parts_a[:12])
            _train(step, range(7, 13), cams, gt, gt_depth, parts)
            _assert_bit_equal(run_a, step, parts_a, parts)
    finally:
        engine.config.deterministic = saved


@pytest.mark.gpu
def test_save_right_after_densification_keeps_the_skipped_step(tmp_path):
    """The skip densify_and_prune arms is state: after a load the model's next optimizer_step is still a no-op (no update,
    no step count), as in the uninterrupted run, and the one after that steps again."""
    step, cam, vm, pm, gt, gt_depth = _make_step(N=12_000)
    step.attach_optimizer("dynamic", ro.GaussianLRs(scaling_lr=0.001, motion_coeff_lr=1.6e-4))
    step.enable_densification("dynamic")
    bt = step.p("table")[cam.time_index].clone()
    for it in range(1, 4):
        step.forward_backward(vm, pm, cam.tanfovx, cam.tanfovy, bt, gt, gt_depth)
        step.add_densification_stats("dynamic")
        step.optimizer_step("dynamic", it)
    st = step.stats["dynamic"]
    thr = float(torch.quantile((st.grad_accum / st.denom.clamp(min=1))[st.denom > 0], 0.7))
    step.densify_and_prune("dynamic", thr, 0.005, 4.0, None, generator=torch.Generator(device="cuda").manual_seed(0))
    step.save(tmp_path / "s.pt")
    back = SplatTrainStep.from_state_dict(torch.load(tmp_path / "s.pt", weights_only=True))
    for s in (step, back):
        before = s.params.clone()
        s.forward_backward(vm, pm, cam.tanfovx, cam.tanfovy, bt, gt, gt_depth)
        assert s.optimizer_step("dynamic", 4) is None
        assert s.optim["dynamic"].steps == 3 and torch.equal(s.params, before)
        s.forward_backward(vm, pm, cam.tanfovx, cam.tanfovy, bt, gt, gt_depth)
        s.optimizer_step("dynamic", 5)
        assert s.optim["dynamic"].steps == 4 and not torch.equal(s.params, before)


@pytest.mark.gpu
def test_exported_models_render_what_the_step_renders():
    """export_models -> render_dynamic (the reference-named tensors, B(t) and the table of the step) == the step's own
    forward: the same kernels on the same inputs."""
    from rodygs_b200.dynamic import GaussianParams, render_dynamic
    from rodygs_b200.rasterizer import GaussianRasterizationSettings
    step, cam, vm, pm, gt, gt_depth = _make_step()
    step.p("basis_t").copy_(step.p("table")[cam.time_index])
    step.forward_backward(vm, pm, cam.tanfovx, cam.tanfovy, step.p("basis_t"), None, None, forward_only=True)
    color, depth, alpha, radii = (t.clone() for t in step.last_outputs)
    d = ck.export_models(step)

    def gp(m):
        return GaussianParams(m["_xyz"], m["_features_dc"], m["_features_rest"], m["_scaling"], m["_rotation"], m["_opacity"])

    settings = GaussianRasterizationSettings(step.H, step.W, cam.tanfovx, cam.tanfovy, step.bg, 1.0, pm, step.sh_degree)
    dyn = d["dynamic"]
    out = render_dynamic(gp(d["static"]), gp(dyn), settings, vm, motion_coeff=dyn["_motion_coeff"],
                         basis_t=d["motion"]["basis_t"], table=d["motion"]["table"], time_ind=dyn["gaussian_to_time_ind"],
                         spatial_lr_scale=d["motion"]["spatial_lr_scale"])
    assert torch.equal(out["radii"], radii) and int((radii > 0).sum()) > 1000
    for name, want in (("rendered_image", color), ("rendered_depth", depth), ("rendered_alpha", alpha)):
        assert float((out[name].detach() - want).abs().max()) <= 1e-6, name


@pytest.mark.gpu
def test_imported_models_build_the_same_flat_parameters():
    step, cam, vm, pm, gt, gt_depth = _make_step()
    step.p("basis_t").copy_(step.p("table")[2])
    again = SplatTrainStep(ck.import_models(ck.export_models(step)), step.H, step.W, sh_degree=3)
    assert again.layout == step.layout
    assert torch.equal(again.params, step.params) and torch.equal(again.time_ind, step.time_ind)


def _digest(t):
    return hashlib.sha256(t.detach().cpu().numpy().tobytes()).hexdigest()


def _dp_resume_worker(rank, world, port, path, ret):
    """Two ranks on ONE GPU over gloo, deterministic backward.  Each rank renders its own views and adds its own
    densification statistics; they are only all-reduced inside densify_and_prune.  The run densifies at step 3, every
    rank saves after step 5 (statistics half accumulated, different on each rank), then the run goes on to the next
    densification at step 7 and one more step - once uninterrupted, once from the file loaded into a step of another
    size on every rank.  Returns what both runs ended with."""
    import os
    import torch.distributed as dist
    from rodygs_b200 import engine
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    engine.config.deterministic = True
    try:
        H, W = 96, 128
        step, cam, vm, pm, gt, gt_depth = _make_step(N=12_000, H=H, W=W)
        step.attach_optimizer("dynamic", ro.GaussianLRs(scaling_lr=0.001, motion_coeff_lr=1.6e-4))
        step.enable_densification("dynamic")

        def dp_step(s, it):
            c = synthetic.make_camera(2 * it + rank, 8, H, W, 6)       # every rank sees different views
            bt = s.p("table")[c.time_index].clone()
            s.forward_backward(c.world_view_transform.t().contiguous().cuda(), c.projection_matrix.t().contiguous().cuda(),
                               c.tanfovx, c.tanfovy, bt, gt, None)
            s.add_densification_stats("dynamic")
            s.allreduce_grads(scale=1.0 / world)
            s.optimizer_step("dynamic", it)

        def densify(s):
            st = s.stats["dynamic"]
            thr = torch.tensor([0.5 * float((st.grad_accum / st.denom.clamp(min=1))[st.denom > 0].mean())], dtype=torch.float64)
            dist.broadcast(thr, 0)
            return s.densify_and_prune("dynamic", float(thr), 0.005, 4.0, None,
                                       generator=torch.Generator(device="cuda").manual_seed(0))

        def finish(s):
            for it in (6, 7):
                dp_step(s, it)
            info = densify(s)
            dp_step(s, 8)
            return (s.nd, info["clones"], info["split_selected"], s.optim["dynamic"].steps, _digest(s.params),
                    _digest(s.optim["dynamic"].exp_avg), _digest(s.optim["dynamic"].exp_avg_sq))

        for it in (1, 2, 3):
            dp_step(step, it)
        densify(step)
        for it in (4, 5):
            dp_step(step, it)
        local = float(step.stats["dynamic"].grad_accum.double().sum())
        step.save(path)
        fresh, *_ = _make_step(N=6_000 + 2_000 * rank, H=H, W=W, seed=rank)
        fresh.load(path)
        same_stats = all(torch.equal(getattr(fresh.stats["dynamic"], f), getattr(step.stats["dynamic"], f))
                         for f in ("grad_accum", "denom", "max_radii2D"))
        ret.put((rank, local, same_stats, finish(step), finish(fresh)))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_data_parallel_resume_between_densifications_matches_the_uninterrupted_run(tmp_path):
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    path = str(tmp_path / "dp.pt")
    procs = [ctx.Process(target=_dp_resume_worker, args=(r, 2, port, path, ret)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([ret.get(timeout=300), ret.get(timeout=300)])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    a, b = res
    assert a[1] != b[1], "the ranks were supposed to hold different statistics when they saved"
    assert a[2] and b[2], "a rank did not get its own statistics back"
    for r in (a, b):
        assert r[4] == r[3], f"rank {r[0]}: the resumed run densified or trained differently: {r[4]} vs {r[3]}"
        # 8 steps minus the two skipped ones after the densifications at steps 3 and 7
        assert r[3][3] == 6 and r[3][1] + r[3][2] > 0
    assert a[3] == b[3], "ranks diverged"
