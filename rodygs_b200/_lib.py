"""ctypes binding of librodygs_b200.so (the C ABI in include/rodygs_b200.h).

There is no CPU fallback: if the shared library is missing or cannot be
loaded, importing the product path raises immediately.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librodygs_b200.so")

c_float_p = C.c_void_p  # raw device pointers travel as integers
c_ptr = C.c_void_p


class RdgSet(C.Structure):
    _fields_ = [("xyz", c_ptr), ("scaling", c_ptr), ("rotation", c_ptr), ("opacity", c_ptr),
                ("sh_dc", c_ptr), ("sh_rest", c_ptr), ("sh_dc_stride", C.c_int32), ("sh_rest_stride", C.c_int32)]


class RdgScene(C.Structure):
    _fields_ = [("n_static", C.c_int64), ("n_dynamic", C.c_int64), ("st", RdgSet), ("dy", RdgSet),
                ("raw", C.c_int32), ("colors_precomp", c_ptr), ("use_deform", C.c_int32),
                ("num_basis", C.c_int32), ("num_times", C.c_int32), ("motion_coeff", c_ptr),
                ("time_ind", c_ptr), ("basis_t", c_ptr), ("table", c_ptr), ("spatial_lr_scale", C.c_float),
                ("frame_order", c_ptr), ("frame_offsets", c_ptr)]


class RdgView(C.Structure):
    _fields_ = [("height", C.c_int32), ("width", C.c_int32), ("tanfovx", C.c_float), ("tanfovy", C.c_float),
                ("scale_modifier", C.c_float), ("sh_degree", C.c_int32), ("enable_cov_grad", C.c_int32),
                ("enable_sh_grad", C.c_int32), ("viewmatrix", c_ptr), ("projmatrix", c_ptr), ("bg", c_ptr)]


class RdgGeom(C.Structure):
    _fields_ = [("radii", c_ptr), ("tiles_touched", c_ptr), ("p0", c_ptr), ("p1", c_ptr), ("p2", c_ptr),
                ("clamped", c_ptr), ("dbg_activated", c_ptr), ("tile_count", c_ptr)]


class RdgBins(C.Structure):
    _fields_ = [("keys_sorted", c_ptr), ("vals_sorted", c_ptr), ("ranges", c_ptr), ("point_offsets", c_ptr),
                ("num_rendered", c_ptr), ("keys_unsorted", c_ptr), ("vals_unsorted", c_ptr), ("region_ids", c_ptr), ("region_masks", c_ptr),
                ("region_count", c_ptr), ("region_stride", C.c_int64)]


class RdgImage(C.Structure):
    _fields_ = [("color", c_ptr), ("depth", c_ptr), ("alpha", c_ptr), ("final_T", c_ptr), ("n_contrib", c_ptr)]


class RdgSetGrad(C.Structure):
    _fields_ = [("xyz", c_ptr), ("scaling", c_ptr), ("rotation", c_ptr), ("opacity", c_ptr),
                ("sh_dc", c_ptr), ("sh_rest", c_ptr)]


class RdgSceneGrad(C.Structure):
    _fields_ = [("st", RdgSetGrad), ("dy", RdgSetGrad), ("colors_precomp", c_ptr), ("means2D", c_ptr),
                ("viewmatrix", c_ptr), ("motion_coeff", c_ptr), ("table", c_ptr), ("basis_t", c_ptr), ("g7_scratch", c_ptr),
                ("models", C.c_int32), ("part", C.c_int32), ("parts", C.c_int32), ("dtable_mode", C.c_int32),
                ("sm_queue", c_ptr), ("dcolor", c_ptr)]


class RdgDensifyField(C.Structure):
    _fields_ = [("src", c_ptr), ("dst", c_ptr), ("width", C.c_int32), ("mode", C.c_int32)]


class RdgShAdam(C.Structure):
    _fields_ = [("exp_avg_dc", c_ptr), ("exp_avg_sq_dc", c_ptr), ("exp_avg_rest", c_ptr), ("exp_avg_sq_rest", c_ptr),
                ("lr_dc", C.c_float), ("lr_rest", C.c_float), ("step", C.c_int32), ("reserved", C.c_int32)]


class RdgAdamGroup(C.Structure):
    _fields_ = [("begin", C.c_int64), ("end", C.c_int64), ("lr", C.c_float), ("reserved", C.c_int32)]


class RdgLossTerms(C.Structure):
    _fields_ = [("depth", c_ptr), ("gt_depth", c_ptr), ("w_pearson", C.c_float), ("pearson_eps", C.c_float),
                ("dL_ddepth", c_ptr), ("alpha", c_ptr), ("w_alpha", C.c_float), ("dL_dalpha", c_ptr),
                ("local_boxes", c_ptr), ("n_local_boxes", C.c_int32), ("w_local", C.c_float)]


class RdgBasisMlp(C.Structure):
    _fields_ = [("emb_dim", C.c_int32), ("width", C.c_int32), ("num_basis", C.c_int32), ("out_dim", C.c_int32),
                ("activation", C.c_int32), ("rows", C.c_int32), ("params", c_ptr), ("emb", c_ptr), ("times", c_ptr),
                ("freqs_pi", c_ptr), ("basis", c_ptr), ("basis_row0", c_ptr), ("saved", c_ptr)]


class RdgRigidity(C.Structure):
    _fields_ = [("n", C.c_int64), ("K", C.c_int32), ("num_basis", C.c_int32), ("n_frames", C.c_int32),
                ("mode_surface", C.c_int32), ("mode_distance", C.c_int32), ("eps", C.c_float),
                ("points", c_ptr), ("canon", c_ptr), ("coeff", c_ptr), ("table", c_ptr), ("frame_indices", c_ptr),
                ("nn_idx", c_ptr), ("nn_dist2", c_ptr), ("loss_parts", c_ptr), ("d_points", c_ptr), ("d_canon", c_ptr),
                ("d_coeff", c_ptr), ("d_table", c_ptr)]


# every symbol include/rodygs_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "rdg_abi_version": (C.c_int, []),
    "rdg_last_error": (C.c_char_p, []),
    "rdg_launch_count": (C.c_uint64, []),
    "rdg_set_tunable": (C.c_int, [C.c_char_p, C.c_int32]),
    "rdg_alpha_reg": (C.c_int, [c_ptr, C.c_int64, C.c_float, c_ptr, c_ptr, c_ptr]),
    "rdg_preprocess_fwd": (C.c_int, [C.POINTER(RdgScene), C.POINTER(RdgView), C.POINTER(RdgGeom), c_ptr]),
    "rdg_bin_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int64, C.c_int32, C.c_int32]),
    "rdg_bin": (C.c_int, [C.c_int64, C.POINTER(RdgGeom), C.c_int32, C.c_int32, C.c_int64, C.POINTER(RdgBins),
                          c_ptr, C.c_int64, c_ptr]),
    "rdg_bin_tiles_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int64, C.c_int32, C.c_int32]),
    "rdg_bin_tiles": (C.c_int, [C.c_int64, C.POINTER(RdgGeom), C.c_int32, C.c_int32, C.c_int64, C.POINTER(RdgBins),
                                c_ptr, C.c_int64, c_ptr]),
    "rdg_blend_fwd": (C.c_int, [C.c_int64, C.POINTER(RdgGeom), C.POINTER(RdgBins), C.POINTER(RdgView),
                                C.POINTER(RdgImage), c_ptr]),
    "rdg_blend_bwd": (C.c_int, [C.c_int64, C.POINTER(RdgGeom), C.POINTER(RdgBins), C.POINTER(RdgView),
                                C.POINTER(RdgImage), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "rdg_blend_bwd_deterministic_scratch_bytes": (C.c_int64, [C.c_int64]),
    "rdg_blend_bwd_deterministic": (C.c_int, [C.c_int64, C.POINTER(RdgGeom), C.POINTER(RdgBins), C.POINTER(RdgView),
                                              C.POINTER(RdgImage), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int64, c_ptr]),
    "rdg_preprocess_bwd": (C.c_int, [C.POINTER(RdgScene), C.POINTER(RdgView), C.POINTER(RdgGeom), c_ptr,
                                     C.POINTER(RdgSceneGrad), c_ptr]),
    "rdg_dcolor_from_acc": (C.c_int, [C.c_int64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "rdg_dcolor_multicast": (C.c_int, [C.c_int64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "rdg_sh_grad_views": (C.c_int, [C.POINTER(RdgScene), C.c_int32, C.c_int32, c_ptr, c_ptr, c_ptr, C.c_float,
                                    C.POINTER(RdgSetGrad), C.POINTER(RdgSetGrad), c_ptr, c_ptr]),
    "rdg_sh_adam_views": (C.c_int, [C.POINTER(RdgScene), C.c_int32, C.c_int32, c_ptr, c_ptr, c_ptr, C.c_float,
                                    C.POINTER(RdgShAdam), C.POINTER(RdgShAdam), C.c_float, C.c_float, C.c_float, c_ptr]),
    "rdg_allreduce_multimem": (C.c_int, [c_ptr, C.c_int64, C.c_int32, C.c_int32, C.c_float, C.c_int32, c_ptr]),
    "rdg_allreduce_multimem_ranges": (C.c_int, [c_ptr, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int32, C.c_int32, C.c_int32,
                                                C.c_float, C.c_int32, c_ptr]),
    "rdg_l1_dssim_workspace_bytes": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "rdg_l1_dssim": (C.c_int, [c_ptr, c_ptr, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float, c_ptr, c_ptr,
                               c_ptr, C.c_int64, c_ptr]),
    "rdg_losses": (C.c_int, [c_ptr, c_ptr, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float, C.POINTER(RdgLossTerms),
                             c_ptr, c_ptr, c_ptr, C.c_int64, c_ptr]),
    "rdg_pearson": (C.c_int, [c_ptr, c_ptr, C.c_int32, C.c_int32, c_ptr, c_ptr, C.c_int32, C.c_float, c_ptr, c_ptr,
                              c_ptr, c_ptr]),
    "rdg_adam": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float,
                           C.c_int32, C.c_float, c_ptr]),
    "rdg_adam_groups": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.POINTER(RdgAdamGroup), C.c_int32, C.c_float, C.c_float,
                                  C.c_float, C.c_int32, C.c_float, c_ptr]),
    "rdg_densify_stats": (C.c_int, [C.c_int64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "rdg_densify_workspace_bytes": (C.c_int64, [C.c_int64]),
    "rdg_densify_plan": (C.c_int, [C.c_int64, c_ptr, C.c_int32, c_ptr, c_ptr, c_ptr, C.c_float, C.c_float, C.c_float,
                                   C.c_float, C.c_int32, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int64, c_ptr]),
    "rdg_densify_apply": (C.c_int, [C.c_int64, c_ptr, c_ptr, c_ptr, c_ptr, C.POINTER(RdgDensifyField), C.c_int32, c_ptr,
                                    c_ptr, C.c_int32, c_ptr, c_ptr]),
    "rdg_reset_opacity": (C.c_int, [C.c_int64, c_ptr, C.c_float, c_ptr, c_ptr, c_ptr]),
    "rdg_motion_coeff_reg": (C.c_int, [C.c_int64, C.c_int32, c_ptr, C.c_float, C.c_float, c_ptr, c_ptr, C.c_int32, c_ptr,
                                       c_ptr]),
    "rdg_motion_basis_reg": (C.c_int, [C.c_int32, C.c_int32, c_ptr, c_ptr, C.c_int32, C.c_int32, C.c_float, c_ptr, c_ptr,
                                       c_ptr, c_ptr]),
    "rdg_knn_workspace_bytes": (C.c_int64, [C.c_int64]),
    "rdg_knn": (C.c_int, [C.c_int64, c_ptr, C.c_int32, c_ptr, c_ptr, c_ptr, C.c_int64, c_ptr]),
    "rdg_knn3_mean_dist2": (C.c_int, [C.c_int64, c_ptr, c_ptr, c_ptr, C.c_int64, c_ptr]),
    "rdg_knn_dist2_bwd": (C.c_int, [C.c_int64, C.c_int32, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "rdg_rigidity_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32]),
    "rdg_rigidity": (C.c_int, [C.POINTER(RdgRigidity), c_ptr, C.c_int64, c_ptr]),
    "rdg_rigidity_sample": (C.c_int, [C.c_int64, C.c_int32, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_float, c_ptr, c_ptr,
                                      c_ptr, c_ptr]),
    "rdg_rigidity_sample_bwd": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_float,
                                          C.c_float, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "rdg_basis_mlp_param_count": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "rdg_basis_mlp_saved_floats": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "rdg_basis_mlp_fwd": (C.c_int, [C.POINTER(RdgBasisMlp), c_ptr]),
    "rdg_basis_mlp_bwd_workspace_bytes": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "rdg_basis_mlp_bwd": (C.c_int, [C.POINTER(RdgBasisMlp), c_ptr, c_ptr, c_ptr, C.c_int32, c_ptr, C.c_int64, c_ptr]),
}

_lib = None


def load() -> C.CDLL:
    """Load the CUDA library (once). Raises if it is not built - there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("RDG_LIB_PATH", LIB_PATH)   # development: an A/B build of the same sources (tools/build_variant.py)
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing. Build it with `python -m rodygs_b200.build` (needs nvcc); "
            "rodygs_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    if lib.rdg_abi_version() != 8:
        raise RuntimeError("librodygs_b200.so ABI version mismatch")
    _lib = lib
    return lib


def set_tunable(name: str, value: int) -> None:
    """A/B switches / test knobs of the launchers (include/rodygs_b200.h: rdg_set_tunable)."""
    check(load().rdg_set_tunable(name.encode(), int(value)))


def check(rc: int) -> None:
    if rc != 0:
        msg = load().rdg_last_error()
        raise RuntimeError(f"rodygs_b200 error {rc}: {msg.decode() if msg else ''}")


def ptr(t):
    """Device pointer of a tensor (or None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr() -> int:
    """cudaStream_t of torch's current stream on the current device.  torch.cuda.current_stream() costs ~15 us per call
    (device lookups, object construction) and the hot path asks four times per step; the raw accessor is ~0.3 us."""
    raw = getattr(torch._C, "_cuda_getCurrentRawStream", None)
    if raw is not None:
        return raw(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors):
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("rodygs_b200 runs on CUDA tensors only (no CPU fallback)")
        if t.dtype not in (torch.float32, torch.int32, torch.int64, torch.uint8):
            raise RuntimeError(f"unsupported dtype {t.dtype}")
