"""3D Gaussian Splatting's PLY file: the one format every Gaussian-splatting viewer reads (INTEGRATION.md §11).

`write_ply(path, records)` writes the records of `SplatTrainStep.export_3dgs` (or any [N, 62] float32 array in the order of
`PLY_PROPERTIES`) as the binary little-endian file that 3DGS's `GaussianModel.save_ply` writes: the same header, the same
property names in the same order (`construct_list_of_attributes`), float32 everywhere.

`read_ply(path)` reads such a file back into the dict `checkpoint.export_models` returns, with the file as the static model:
`checkpoint.import_models(read_ply(path))` is a scene `SplatTrainStep` takes.  Host code only, no `plyfile` dependency.
"""
from __future__ import annotations

import os
from typing import Dict, List, Union

import numpy as np
import torch

PLY_PROPERTIES: List[str] = (["x", "y", "z", "nx", "ny", "nz"] + [f"f_dc_{i}" for i in range(3)]
                             + [f"f_rest_{i}" for i in range(45)] + ["opacity"] + [f"scale_{i}" for i in range(3)]
                             + [f"rot_{i}" for i in range(4)])
RECORD_FLOATS = len(PLY_PROPERTIES)            # 62: 248 bytes per Gaussian
REQUIRED = ["x", "y", "z", "f_dc_0", "f_dc_1", "f_dc_2", "opacity", "scale_0", "scale_1", "scale_2",
            "rot_0", "rot_1", "rot_2", "rot_3"]
FLOAT_TYPES = ("float", "float32")
NUM_BASIS = 16                                 # the zero motion table of a file read as a static scene: [1, 16, 7]


def ply_header(n: int) -> bytes:
    """The header 3DGS's save_ply writes for n Gaussians (plyfile's layout, no comment lines)."""
    lines = ["ply", "format binary_little_endian 1.0", f"element vertex {int(n)}"]
    lines += [f"property float {name}" for name in PLY_PROPERTIES]
    lines.append("end_header")
    return ("\n".join(lines) + "\n").encode("ascii")


def write_ply(path: Union[str, os.PathLike], records) -> None:
    """Write records [N, 62] float32 (a tensor on any device, or a numpy array) as a 3DGS PLY file.  A device tensor is
    copied to the host first (N x 248 bytes of host memory)."""
    if torch.is_tensor(records):
        if records.dtype != torch.float32:
            raise ValueError(f"write_ply: records must be float32, got {records.dtype}")
        records = records.detach().cpu().numpy()
    arr = np.asarray(records)
    if arr.dtype != np.float32 or arr.ndim != 2 or arr.shape[1] != RECORD_FLOATS:
        raise ValueError(f"write_ply: records must be a float32 array of shape [N, {RECORD_FLOATS}], got {arr.dtype} "
                         f"{arr.shape}")
    arr = np.ascontiguousarray(arr, dtype="<f4")
    with open(path, "wb") as f:
        f.write(ply_header(arr.shape[0]))
        arr.tofile(f)


def _parse_header(f, path) -> tuple:
    """(vertex count, vertex property names) of a binary little-endian PLY file whose first element is `vertex` with float
    properties only; f is left at the first byte of the body."""
    if f.readline().rstrip(b"\r\n") != b"ply":
        raise ValueError(f"read_ply: {path} is not a PLY file (no 'ply' magic line)")
    fmt, n, props, elements = None, None, [], 0
    while True:
        raw = f.readline()
        if not raw:
            raise ValueError(f"read_ply: {path}: the header has no end_header line")
        words = raw.decode("ascii", errors="replace").split()
        if not words or words[0] in ("comment", "obj_info"):
            continue
        if words[0] == "end_header":
            break
        if words[0] == "format":
            fmt = " ".join(words[1:])
            if words[1:2] != ["binary_little_endian"]:
                raise ValueError(f"read_ply: {path} is '{fmt}'; only binary_little_endian files are read")
        elif words[0] == "element":
            elements += 1
            if elements == 1:
                if len(words) != 3 or words[1] != "vertex":
                    raise ValueError(f"read_ply: {path}: the first element is '{' '.join(words[1:])}', not 'vertex'")
                n = int(words[2])
                if n < 0:
                    raise ValueError(f"read_ply: {path}: negative vertex count {n}")
        elif words[0] == "property":
            if elements == 1:
                if words[1] == "list" or words[1] not in FLOAT_TYPES or len(words) != 3:
                    raise ValueError(f"read_ply: {path}: vertex property '{' '.join(words[1:])}' is not float; only "
                                     "float32 properties are read")
                props.append(words[2])
        else:
            raise ValueError(f"read_ply: {path}: unknown header line '{' '.join(words)}'")
    if fmt is None:
        raise ValueError(f"read_ply: {path}: the header has no format line")
    if n is None:
        raise ValueError(f"read_ply: {path}: no vertex element")
    return n, props


def read_ply(path: Union[str, os.PathLike]) -> Dict[str, Dict]:
    """A 3DGS PLY file as export_models' dict, the file as the static model: {"static": {"_xyz" [n,3], "_scaling" [n,3],
    "_rotation" [n,4], "_opacity" [n,1], "_features_dc" [n,1,3], "_features_rest" [n,15,3]}, "dynamic": the same with 0
    rows + "_motion_coeff" [0,1,16] and "gaussian_to_time_ind" [0], "motion": {"table": zeros [1,16,7], "basis_t": zeros
    [16,7], "spatial_lr_scale": 1.0}}; CPU float32 tensors.

    Properties are found by name; others (normals, extra attributes) are ignored.  f_rest_* of files of SH degree 0-2
    (0, 9 or 24 of them, channel-major like degree 3's 45) fill the first coefficients and the rest are 0.  Refused with a
    ValueError naming the problem: ascii or big-endian files, non-float vertex properties, a missing required property,
    a first element that is not `vertex`, and a body shorter than the header says."""
    with open(path, "rb") as f:
        n, props = _parse_header(f, path)
        missing = [p for p in REQUIRED if p not in props]
        if missing:
            raise ValueError(f"read_ply: {path} lacks the required properties {missing}")
        rest = [p for p in props if p.startswith("f_rest_")]
        if len(rest) not in (0, 9, 24, 45) or sorted(rest) != sorted(f"f_rest_{i}" for i in range(len(rest))):
            raise ValueError(f"read_ply: {path}: f_rest_* must be f_rest_0..f_rest_{{8, 23, 44}} (SH degree 1-3) or "
                             f"absent, got {len(rest)} of them")
        count = n * len(props)
        body = np.fromfile(f, dtype="<f4", count=count)
    if body.size < count:
        raise ValueError(f"read_ply: {path}: the body holds {body.size * 4} bytes, the header says {count * 4} "
                         f"({n} vertices x {len(props)} float properties)")
    table = body.reshape(n, len(props))
    col = {name: i for i, name in enumerate(props)}

    def cols(names):
        return torch.from_numpy(np.ascontiguousarray(table[:, [col[c] for c in names]], dtype=np.float32))

    R = len(rest) // 3                      # higher-order coefficients in the file, stored channel-major: f_rest_{c R + j}
    features_rest = torch.zeros(n, 15, 3, dtype=torch.float32)
    if R:
        features_rest[:, :R, :] = cols([f"f_rest_{c * R + j}" for c in range(3) for j in range(R)]).view(n, 3, R).transpose(1, 2)
    static = {"_xyz": cols(["x", "y", "z"]), "_scaling": cols(["scale_0", "scale_1", "scale_2"]),
              "_rotation": cols(["rot_0", "rot_1", "rot_2", "rot_3"]), "_opacity": cols(["opacity"]),
              "_features_dc": cols(["f_dc_0", "f_dc_1", "f_dc_2"]).view(n, 1, 3), "_features_rest": features_rest}
    dynamic = {k: v.new_zeros((0,) + tuple(v.shape[1:])) for k, v in static.items()}
    dynamic["_motion_coeff"] = torch.zeros(0, 1, NUM_BASIS)
    dynamic["gaussian_to_time_ind"] = torch.zeros(0, dtype=torch.int64)
    motion = {"table": torch.zeros(1, NUM_BASIS, 7), "basis_t": torch.zeros(NUM_BASIS, 7), "spatial_lr_scale": 1.0}
    return {"static": static, "dynamic": dynamic, "motion": motion}
