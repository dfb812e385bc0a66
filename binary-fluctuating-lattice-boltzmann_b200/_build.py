"""Build recipe for the CUDA library (sm_100a only; nvcc cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbflbm.so")
SOURCES = ["capi.cu", "multi.cu"]
HEADERS = ["d3q19.cuh", "philox.cuh", "physics.cuh", "kernels.cuh", "fused.cuh"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "--shared", "-Xcompiler", "-fPIC",
]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.join(HERE, "..", "include", "bflbm.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


SF_LIB = os.path.join(HERE, "libbflbm_sf.so")


def build_sf(force: bool = False) -> str:
    """Compile csrc/sf.cu and csrc/sf_slab.cu (on-GPU structure-factor accumulators, cuFFT) into libbflbm_sf.so on top of
    libbflbm.so."""
    build()
    srcs = [os.path.join(CSRC, s) for s in ("sf.cu", "sf_slab.cu")]
    deps = srcs + [LIB, os.path.join(CSRC, "sf_common.cuh")] + \
        [os.path.join(HERE, "..", "include", h) for h in ("bflbm_sf.h", "bflbm_sf_slab.h")]
    if not force and os.path.exists(SF_LIB) and all(os.path.getmtime(d) <= os.path.getmtime(SF_LIB) for d in deps):
        return SF_LIB
    cmd = [nvcc()] + NVCC_FLAGS + srcs + ["-o", SF_LIB, "-L" + HERE, "-lbflbm", "-lcufft", "-Xlinker", "-rpath,$ORIGIN"]
    subprocess.run(cmd, check=True)
    return SF_LIB


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/ into libbflbm.so next to this file (in-tree, so it travels with the repo)."""
    if not force and not needs_build():
        return LIB
    cmd = [nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB]
    subprocess.run(cmd, check=True)
    return LIB
