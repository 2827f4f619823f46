"""Builds ``libcistaflow.so`` in-tree with nvcc for sm_100a (B200).

No torch dependency: the library is plain CUDA C++ behind the C ABI of
``include/cistaflow.h``.  nvcc cross-compiles without a GPU, so this is also
the "does it build" check that ``__graft_entry__.build()`` runs on CPU.
The built ``.so`` is git-ignored but travels with the gpurun snapshot.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB = os.path.join(HERE, "libcistaflow.so")
STAMP = os.path.join(HERE, ".libcistaflow.stamp")

HEADERS = ["cistaflow.h", "cistaflow_altcorr.h", "cistaflow_det.h", "cistaflow_half.h"]
SOURCES = ["api.cu", "voxel.cu", "voxel_tiled.cu", "voxel_packed.cu", "warp.cu", "warp_tma.cu", "warp_backward.cu", "warp_backward_det.cu", "fwl.cu", "corr_lookup.cu", "corr_lookup_backward.cu", "corr_build.cu", "corr_build_tc.cu", "corr_alt.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "-shared", "-cudart", "static",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _fingerprint() -> str:
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(INCLUDE, h) for h in HEADERS]
    for f in files:
        h.update(f.encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile if sources changed; returns the path of the shared library."""
    fp = _fingerprint()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == fp:
        return LIB
    cmd = [_nvcc(), *NVCC_FLAGS, "-I", INCLUDE, "-I", CSRC, "-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
        print(" ".join(cmd), file=sys.stderr)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose:
        sys.stderr.write(res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    with open(STAMP, "w") as fh:
        fh.write(fp)
    return LIB


def build_variant(name: str, defines: list[str]) -> str:
    """Experiment builds (scripts/): the same sources with extra -D flags, written to
    build/libcistaflow_<name>.so and loaded through the CISTAFLOW_LIB environment variable."""
    out_dir = os.path.join(ROOT, "build")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, f"libcistaflow_{name}.so")
    cmd = [_nvcc(), *NVCC_FLAGS, *[f"-D{d}" for d in defines], "-I", INCLUDE, "-I", CSRC, "-o", out] + \
        [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
