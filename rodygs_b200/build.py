"""In-tree build of librodygs_b200.so for sm_100a with plain nvcc.

No torch / pybind dependency: the library is a C-ABI shared object
(include/rodygs_b200.h) that rodygs_b200/_lib.py loads with ctypes.

    python -m rodygs_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ_DIR = os.path.join(HERE, "_build")
LIB_PATH = os.path.join(HERE, "librodygs_b200.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
          "--expt-relaxed-constexpr"]
# Translation units whose float results feed integer outputs (depth bits -> sort keys,
# radius / pixel centre -> tile rectangle) are built without FMA contraction so that
# they are bit-identical to the oracle's individually rounded float32 operations.
SOURCES = {
    "api.cu": [],
    "preprocess_fwd.cu": ["-fmad=false"],
    "binning.cu": ["-fmad=false"],
    "binning_tiles.cu": ["-fmad=false"],
    "blend.cu": [],
    "preprocess_bwd.cu": [],
    "sh_grad_views.cu": [],
    "exchange.cu": [],
    "loss.cu": [],
    "densify.cu": [],
    "optim.cu": [],
    "motion_reg.cu": [],
    "knn.cu": ["-fmad=false"],
    "rigidity.cu": [],
    "basis_mlp.cu": [],
    "metrics.cu": [],
    "pose.cu": [],
    "lpips.cu": [],
    "track.cu": ["-fmad=false"],
}
# every header the sources include takes part in the digest, so that editing one rebuilds the library
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith(".cuh")) + [os.path.join("..", "..", "include", "rodygs_b200.h")]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; rodygs_b200 has no CPU fallback and cannot be built without CUDA")


def _digest() -> str:
    h = hashlib.sha256()
    for name in sorted(SOURCES) + HEADERS + [os.path.basename(__file__)]:
        path = os.path.join(CSRC, name) if name != os.path.basename(__file__) else os.path.abspath(__file__)
        with open(path, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every kernel for sm_100a and link the shared library. Returns its path."""
    os.makedirs(OBJ_DIR, exist_ok=True)
    stamp = os.path.join(OBJ_DIR, "digest.txt")
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp) and open(stamp).read() == digest:
        return LIB_PATH
    nvcc = _nvcc()
    objs = []
    procs = []
    for src, extra in SOURCES.items():
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *ARCH, *COMMON, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0 or verbose:
            print(f"--- {src} ---\n{out}", flush=True)
        failed |= pr.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed (see output above)")
    cmd = [nvcc, *ARCH, "-shared", "-o", LIB_PATH, *objs, "-lcudart"]
    subprocess.run(cmd, check=True)
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB_PATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
