"""Builds cvmatrix_b200/libcvmx.so (C ABI + sm_100a kernels) in-tree with nvcc.

    python -m cvmatrix_b200.build [--force]

The library is compiled for sm_100a only (-gencode arch=compute_100a,code=sm_100a); nvcc
cross-compiles without a GPU.  The static CUDA runtime is linked in, so the .so has no
dependency on torch or on a system libcudart.
"""

from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libcvmx.so")
SOURCES = ["cvmx_api.cu"]
HEADERS = ["host_stager.h", "common.cuh", "kernels_stats.cuh", "kernels_scan.cuh", "kernels_gram.cuh", "kernels_gram_tc.cuh", "kernels_pls.cuh", "kernels_ridge.cuh", os.path.join("..", "..", "include", "cvmx.h")]

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-pthread", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libcvmx.so cannot be built (set NVCC=/path/to/nvcc)")


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_lib(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv))
