"""Builds icet_b200/lib/libicet_b200.so (sm_100a only) with nvcc.  In-tree so that the .so travels
to the GPU box with the repository snapshot."""
from __future__ import annotations

import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIBDIR = os.path.join(_HERE, "lib")
LIB = os.path.join(LIBDIR, "libicet_b200.so")
SOURCES = [os.path.join(CSRC, "icet_b200.cu")]
DEPS = SOURCES + [os.path.join(CSRC, f) for f in ("icet_math.cuh", "synth.h", "chunk.cuh", "kernels_scan1.cuh", "kernels_pass.cuh", "kernels_pass2.cuh", "kernels_loop.cuh", "kernels_cluster.cuh",
                                                 "runtime.inl", "callers.cuh", "callers_abi.inl", "kernels_kfnode.cuh",
                                                 "kfnode_abi.inl", "multi_abi.inl")] + [
    os.path.join(os.path.dirname(_HERE), "include", "icet_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    # no FMA contraction: the point-wise geometry must round like the reference's scalar code
    # (the libm routines use explicit fma intrinsics and are not affected)
    "-fmad=false",
    "-Xcompiler", "-fPIC", "-shared", "-ldl",
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    cmd = [nvcc_path()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
