"""Shared test utilities: scene assembly for the oracle and for the CUDA path."""
import math

import torch

from oracle import deform_oracle as do
from oracle import splat_oracle as so
from rodygs_b200 import synthetic


def small_scene(n=3000, H=96, W=128, T=6, seed=0, radius_px=5.0):
    sc = synthetic.make_scene(n, H, W, T, seed=seed, radius_px=radius_px)
    cam = synthetic.make_camera(1, 4, H, W, T)
    return sc, cam


def raw_sets(sc):
    st = do.RawGaussians(**sc["static"])
    dy = do.RawGaussians(**sc["dynamic"])
    return st, dy


def activated_concat(sc, cam, use_deform=True):
    """Reference chain on the CPU: activations + deformation + concat (oracle)."""
    st, dy = raw_sets(sc)
    basis_t = sc["table"][cam.time_index]
    return do.assemble(st, dy, sc["motion_coeff"].squeeze(1), basis_t, sc["table"], sc["time_ind"].long(),
                       sc["spatial_lr_scale"], use_deform)


def oracle_settings(cam, bg, sh_degree=3, scale_modifier=1.0, cov=True, sh=True):
    return so.Settings(cam.height, cam.width, cam.tanfovx, cam.tanfovy, bg, scale_modifier,
                       cam.projection_matrix.t().contiguous(), sh_degree, False, False, cov, sh)


def rel_err(a, b):
    """max|a-b| / max|b| (norm-wise relative error used for gradients)."""
    denom = b.abs().max().item()
    return (a - b).abs().max().item() / max(denom, 1e-30)


def elementwise_ok(got, ref, rtol=1e-3, floor=1e-5):
    """Element-wise gradient bar |a - b| <= rtol |b| + floor max|b| (a tensor whose small entries are all wrong fails here,
    while it would pass the norm-wise rel_err); returns (ok, worst |a - b| / bound)."""
    got, ref = got.double().cpu(), ref.double().cpu()
    bound = (rtol * ref.abs() + floor * ref.abs().max()).clamp_min(1e-300)
    ratio = ((got - ref).abs() / bound).max().item()
    return ratio <= 1.0, ratio


def elementwise_vs_truth(got, ref32, ref64, rtol=1e-3, floor=1e-5):
    """Element-wise bar against the float64 oracle: |a - b64| <= rtol |b64| + floor max|b64| - or, where float32 arithmetic
    cannot resolve that (sums with cancellation: the float32 ORACLE misses its own float64 twin by more), 1.5 x the float32
    oracle's error.  Returns (ok, ratio of the CUDA result, ratio of the float32 oracle)."""
    got, ref32, ref64 = got.double().cpu(), ref32.double().cpu(), ref64.double().cpu()
    bound = (rtol * ref64.abs() + floor * ref64.abs().max()).clamp_min(1e-300)
    r_cu = ((got - ref64).abs() / bound).max().item()
    r_32 = ((ref32 - ref64).abs() / bound).max().item()
    return r_cu <= max(1.0, 1.5 * r_32), r_cu, r_32
