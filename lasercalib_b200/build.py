"""Build liblcba.so (the C-ABI + sm_100a kernels) in-tree with nvcc.

    python -m lasercalib_b200.build [--force]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels with the tree.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "liblcba.so")
SOURCES = ["lcba.cu"]
HEADERS = ["common.cuh", "model.cuh", "eval.cuh", "ingest.cuh", "linearize.cuh", "schur.cuh", "schur_mma.cuh", "schur_i8.cuh", "peer_reduce.cuh",
           "dense.cuh", "dense_passes.cuh", "control.cuh", "variants.cuh", "bounds.cuh", os.path.join("..", "..", "include", "lcba.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-diag-suppress", "177"]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def is_stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not is_stale():
        return LIB
    cmd = [find_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl"]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout + proc.stderr)
    if verbose:
        print(proc.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
