"""The reference arm of bench.py (CPU only: the oracle on a bounded, density-matched sample of the bench workload) prints
one JSON line that follows the driver's contract.  Uses the smallest workload so that the test stays within seconds."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "c1_cpu",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "it/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 2 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "oracle" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]
    # honest bookkeeping (VERDICT r01): the frames actually run, an explicit extrapolation flag, the workload's own counts
    assert d["extrapolated"] is True and d["warmup"] == 1 and d["requested_steps"] == 2
    wc = d["config"]["workload_counts"]
    assert wc["n"] == 10000 and 0 < wc["visible"] <= wc["n"] and wc["duplicates"] >= wc["visible"]
    assert d["metric"].startswith("train iters/sec (raster fwd+bwd+loss) at 256x256/10K Gaussians")


def test_reference_arm_caps_the_frames_it_runs():
    sys.path.insert(0, ROOT)
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    assert b.metric_name("c4_iphone") == "train iters/sec (raster fwd+bwd+loss) at 1080p/2M Gaussians; % HBM roofline"   # BASELINE.json
    assert "960x540/1M" in b.metric_name("c3_nvidia") and "512x512/300K" in b.metric_name("c2_kubric")
    assert b.sample_shape("c4_iphone")[:3] == (62745, 256, 256)


def test_dump_outputs_writes_the_last_step_within_64_mb(tmp_path):
    """--dump-outputs at the flagship's image size (1080p) with more Gaussians per model than the sample takes (so the same
    bytes as 2M Gaussians): float32 / float64 arrays only, at most 64 MB, the sampled rows are the ones the indices name,
    and the sample is the same from run to run."""
    import importlib.util
    import types

    import numpy as np
    import torch
    spec =importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    from rodygs_b200 import trainer
    ns, nd, K, T, H, W = 20000, 20001, 16, 100, 1080, 1920
    layout, total = trainer.flat_layout(ns, nd, K, T)
    grads = torch.randn(total, generator=torch.Generator().manual_seed(1))
    step = types.SimpleNamespace(ns=ns, nd=nd, loss_parts=torch.rand(8), view_grad=torch.randn(4, 4),
                                 means2D_grad=torch.randn(ns + nd, 3),
                                 last_outputs=(torch.rand(3, H, W), torch.rand(1, H, W), torch.rand(1, H, W),
                                               torch.randint(0, 50, (ns + nd,), dtype=torch.int32)))
    step.g = lambda name: trainer.SplatTrainStep._slice(step, grads, name)
    step.layout = layout
    for run in ("a", "b"):
        b.dump_outputs(step, str(tmp_path / run), forward_only=False, with_sh=True)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b"))
    arrays = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    for f in files:
        assert np.array_equal(arrays[f[:-4]], np.load(tmp_path / "b" / f)), f
    idx = torch.from_numpy(arrays["index_dynamic"]).long()
    assert len(idx) == b.DUMP_ROWS and len(arrays["index_static"]) == b.DUMP_ROWS
    for k in trainer.PARAM_ORDER + ("motion_coeff",):
        ref = step.g(k if k == "motion_coeff" else f"dynamic.{k}")[idx]
        assert np.array_equal(arrays[f"grad_dynamic_{k}"], ref.numpy()), k
    assert np.array_equal(arrays["radii_dynamic"], step.last_outputs[3][ns + idx].float().numpy())
    assert np.array_equal(arrays["grad_means2D_dynamic"], step.means2D_grad[ns + idx].numpy())
    assert arrays["color"].shape == (3, H, W) and arrays["grad_table"].shape == (T, K, 7)


def test_cpu_sample_matches_the_workload_density():
    """The bounded sample keeps the workload's Gaussians per tile: N' = N * 256 / tiles on a 256x256 window."""
    sys.path.insert(0, ROOT)
    from rodygs_b200 import synthetic
    for cfg, (N, H, W, T, _) in synthetic.CONFIGS.items():
        if cfg == "c1_cpu":
            continue
        tiles = ((H + 15) // 16) * ((W + 15) // 16)
        n_sample = int(round(N * 256 / tiles))
        assert abs(n_sample / 256 - N / tiles) < 1.0
        assert n_sample < 200_000            # seconds per frame on the host cores, not minutes
