"""The flat-buffer trainer's models as the reference's parameter tensors, and back.

`export_models(step)` returns the static and the dynamic model under the attribute names of RoDyGS's Gaussian models
(DESIGN.md §3): `_xyz`, `_scaling`, `_rotation`, `_opacity`, `_features_dc [n,1,3]`, `_features_rest [n,15,3]`; the dynamic
model also `_motion_coeff [n,1,K]`, `gaussian_to_time_ind` (int64), `gaussian_to_time` (when the training times are known,
i.e. a basis MLP is attached) and the MLP's reference `state_dict()` under `_deform_network`.  These are the tensors
`rodygs_b200.dynamic.GaussianParams` / `render_dynamic` and the `diff_gauss_pose` drop-in take.  `import_models(d)` is the
inverse: the scene dict `SplatTrainStep(scene, ...)` takes.

Only these names and shapes are assumed.  The reference's checkpoint layout (`rodygs_static.py:321-347`,
`rodygs_dynamic.py:217-222`: which attributes `torch.save` writes, in which container, next to which iteration counter) is
not in this tree, so it is recalled, not pinned: map the dicts into and out of a `.ckpt` file at the call site.

The step holds three things no reference model does: the motion table B(t_i) [T,K,7] (the MLP's output at the training
times, or a free tensor when no MLP is attached), B(t) [K,7] of the last query time and `spatial_lr_scale`.  They travel
under the separate key "motion" so that the round trip is lossless.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from .trainer import PARAM_ORDER

TAGS = ("static", "dynamic")


def export_models(step) -> Dict[str, Dict]:
    """{"static": {...}, "dynamic": {...}, "motion": {"table", "basis_t", "spatial_lr_scale"}}; tensors are copies on the
    step's device (they outlive the next densification, which replaces the flat buffers)."""
    out = {tag: {f"_{k}": step.p(f"{tag}.{k}").detach().clone() for k in PARAM_ORDER} for tag in TAGS}
    dyn = out["dynamic"]
    dyn["_motion_coeff"] = step.p("motion_coeff").detach().clone()
    dyn["gaussian_to_time_ind"] = step.time_ind.to(torch.int64)
    mlp = getattr(step, "mlp", None)
    if mlp is not None:
        train_times = step._mlp_times[1:]
        dyn["gaussian_to_time"] = train_times[step.time_ind.long()].clone()
        dyn["_deform_network"] = mlp.state_dict()
    out["motion"] = {"table": step.p("table").detach().clone(), "basis_t": step.p("basis_t").detach().clone(),
                     "spatial_lr_scale": float(step.spatial_lr_scale)}
    return out


def import_models(d: Dict[str, Dict], table: Optional[torch.Tensor] = None, basis_t: Optional[torch.Tensor] = None,
                  spatial_lr_scale: Optional[float] = None) -> Dict:
    """The scene dict of `SplatTrainStep(scene, ...)` from reference-named tensors (export_models' output or a model the
    reference trained).  table / basis_t / spatial_lr_scale override d["motion"]; without d["motion"] the table is
    required (compute it with `BasisMLP.query_and_table(t, train_times)` after loading `_deform_network`) and
    spatial_lr_scale defaults to 1.  `_deform_network` itself goes to `BasisMLP.load_state_dict` +
    `SplatTrainStep.attach_basis_mlp`."""
    motion = d.get("motion", {})
    table = motion.get("table") if table is None else table
    if table is None:
        raise ValueError("import_models: no motion table - pass table=[T,K,7] (B at every training time)")
    basis_t = motion.get("basis_t") if basis_t is None else basis_t
    if spatial_lr_scale is None:
        spatial_lr_scale = motion.get("spatial_lr_scale", 1.0)
    scene = {}
    for tag in TAGS:
        src = d[tag]
        missing = [f"_{k}" for k in PARAM_ORDER if f"_{k}" not in src]
        if missing:
            raise KeyError(f"import_models: the {tag} model has no {missing}")
        scene[tag] = {k: src[f"_{k}"].detach().to(torch.float32) for k in PARAM_ORDER}
        n = scene[tag]["xyz"].shape[0]
        want = {"xyz": (n, 3), "scaling": (n, 3), "rotation": (n, 4), "opacity": (n, 1), "features_dc": (n, 1, 3),
                "features_rest": (n, 15, 3)}
        for k, shp in want.items():
            if tuple(scene[tag][k].shape) != shp:
                raise ValueError(f"import_models: {tag}._{k} has shape {tuple(scene[tag][k].shape)}, expected {shp}")
    dyn, nd = d["dynamic"], scene["dynamic"]["xyz"].shape[0]
    K = table.shape[1]
    coeff = dyn["_motion_coeff"].detach().to(torch.float32)
    if tuple(coeff.shape) != (nd, 1, K) or tuple(table.shape) != (table.shape[0], K, 7):
        raise ValueError(f"import_models: _motion_coeff {tuple(coeff.shape)} and table {tuple(table.shape)} must be "
                         f"[{nd},1,K] and [T,K,7]")
    ti = dyn["gaussian_to_time_ind"]
    if tuple(ti.shape) != (nd,) or ti.dtype.is_floating_point:
        raise ValueError(f"import_models: gaussian_to_time_ind must be an integer tensor of shape ({nd},)")
    if nd > 0 and (int(ti.min()) < 0 or int(ti.max()) >= table.shape[0]):
        raise ValueError(f"import_models: gaussian_to_time_ind must lie in [0, {table.shape[0]}) (the table's rows)")
    scene.update(motion_coeff=coeff, table=table.detach().to(torch.float32), time_ind=ti.to(torch.int32),
                 spatial_lr_scale=float(spatial_lr_scale))
    if basis_t is not None:
        scene["basis_t"] = basis_t.detach().to(torch.float32)
    return scene
