"""Builds csrc/libgaccum.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libgaccum.so")
SOURCES = ["gaccum_abi.cu"]
# every file the translation unit includes: editing any of them must rebuild libgaccum.so (a stale binary
# travels to the GPU box and silently runs old kernels)
DEPS = SOURCES + sorted(f for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))) + ["../../include/gaccum.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
    "-Xcompiler", "-fPIC,-fvisibility=hidden,-ffp-contract=off,-O2",
    "-cudart", "static",
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libgaccum.so cannot be built (there is no CPU fallback)")


def stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build_libgaccum(force: bool = False, verbose: bool = False) -> str:
    if force or stale():
        cmd = [nvcc_path()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
        env = dict(os.environ)
        env.pop("CC", None); env.pop("CXX", None)   # the image's CC wrapper lacks parts of the toolchain
        subprocess.check_call(cmd, cwd=CSRC, env=env)
    return LIB


if __name__ == "__main__":
    print(build_libgaccum(force=True, verbose=True))
