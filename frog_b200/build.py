"""Build recipes for the native artefacts (in-tree, so the built files travel with `gpurun`).

    frog_b200/libfrogmatch.so   CUDA kernels + C ABI (include/frogmatch.h), sm_100a only
    bin/match                   the drop-in `match` executable (C++ host, links libfrogmatch.so)
    frog_b200/libfrogsurf.so    SURF3D producer (SURVEY 8f-4): CUDA kernels + C ABI (include/frogsurf.h)
    bin/surf3d                  the `surf3d` executable over it (MetaImage volumes in, keypoint files out)

`python -m frog_b200.build` builds both; nvcc cross-compiles sm_100a without a GPU.
"""
from __future__ import annotations

import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "frog_b200", "csrc")
LIB = os.path.join(ROOT, "frog_b200", "libfrogmatch.so")
BIN = os.path.join(ROOT, "bin", "match")
FMIO = os.path.join(ROOT, "frog_b200", "libfmio.so")
SURF_LIB = os.path.join(ROOT, "frog_b200", "libfrogsurf.so")
SURF_BIN = os.path.join(ROOT, "bin", "surf3d")
FSIO = os.path.join(ROOT, "frog_b200", "libfsio.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fopenmp",
]


def _newer(target: str, sources) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _sources(exts):
    out = [os.path.join(ROOT, "include", f) for f in os.listdir(os.path.join(ROOT, "include"))]
    out += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(exts)]
    return out


def build_lib(force: bool = False, verbose: bool = False) -> str:
    srcs = _sources((".cu", ".cuh", ".h"))
    if not force and _newer(LIB, srcs):
        return LIB
    cmd = ["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + [
        "-shared", "-o", LIB, os.path.join(CSRC, "fm_api.cu")]
    subprocess.run(cmd, check=True, cwd=ROOT)
    return LIB


def build_cli(force: bool = False) -> str:
    srcs = _sources((".cpp", ".h"))
    if not force and _newer(BIN, srcs + [LIB]):
        return BIN
    os.makedirs(os.path.dirname(BIN), exist_ok=True)
    cmd = ["g++", "-O2", "-std=c++17", "-fopenmp", "-I", os.path.join(ROOT, "include"),
           os.path.join(CSRC, "match_main.cpp"), os.path.join(CSRC, "keypoint_io.cpp"), os.path.join(CSRC, "fast_inflate.cpp"),
           os.path.join(CSRC, "surf_io.cpp"),
           "-o", BIN, "-L", os.path.dirname(LIB), "-lfrogmatch", "-lz", "-ldl",
           "-Wl,-rpath,$ORIGIN/../frog_b200"]
    # (libfrogsurf.so is not linked: bin/match dlopens it, through the same run path, when a list holds volumes)
    # multi-GPU list gather over NCCL (system libnccl; only the executable links it, never libfrogmatch.so, so a
    # Python process that already carries torch's NCCL is not given a second copy)
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    if os.path.exists("/usr/include/nccl.h") and os.path.exists(os.path.join(cuda, "include", "cuda_runtime.h")):
        cmd += ["-DFM_WITH_NCCL", "-I", os.path.join(cuda, "include"), "-L", os.path.join(cuda, "lib64"), "-lnccl", "-lcudart"]
    subprocess.run(cmd, check=True, cwd=ROOT)
    return BIN


def build_fmio(force: bool = False) -> str:
    """Host-side readers / pruning / pairs.bin writer as a small C library (no CUDA)."""
    srcs = _sources((".cpp", ".h"))
    if not force and _newer(FMIO, srcs):
        return FMIO
    cmd = ["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(ROOT, "include"),
           os.path.join(CSRC, "fmio_capi.cpp"), os.path.join(CSRC, "keypoint_io.cpp"), os.path.join(CSRC, "fast_inflate.cpp"),
           "-o", FMIO, "-lz"]
    subprocess.run(cmd, check=True, cwd=ROOT)
    return FMIO


def build_surf_lib(force: bool = False, verbose: bool = False) -> str:
    srcs = [os.path.join(CSRC, f) for f in ("fs_api.cu", "fs_kernels.cuh", "fs_as_read.cuh")] + [
        os.path.join(ROOT, "include", f) for f in ("frogsurf.h", "frogsurf_debug.h")]
    if not force and _newer(SURF_LIB, srcs):
        return SURF_LIB
    # -fmad=false: the host and device statements of the interpolation solve must execute the same IEEE operations
    cmd = ["nvcc"] + NVCC_FLAGS + ["-fmad=false"] + (["-Xptxas", "-v"] if verbose else []) + [
        "-shared", "-o", SURF_LIB, os.path.join(CSRC, "fs_api.cu")]
    subprocess.run(cmd, check=True, cwd=ROOT)
    return SURF_LIB


def build_surf_cli(force: bool = False) -> str:
    srcs = [os.path.join(CSRC, f) for f in ("surf_main.cpp", "surf_io.cpp", "surf_io.h")] + [os.path.join(ROOT, "include", "frogsurf.h")]
    if not force and _newer(SURF_BIN, srcs + [SURF_LIB]):
        return SURF_BIN
    os.makedirs(os.path.dirname(SURF_BIN), exist_ok=True)
    cmd = ["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"),
           os.path.join(CSRC, "surf_main.cpp"), os.path.join(CSRC, "surf_io.cpp"),
           "-o", SURF_BIN, "-L", os.path.dirname(SURF_LIB), "-lfrogsurf", "-lz", "-Wl,-rpath,$ORIGIN/../frog_b200"]
    subprocess.run(cmd, check=True, cwd=ROOT)
    return SURF_BIN


def build_fsio(force: bool = False) -> str:
    """bin/surf3d's host I/O (MetaImage reader, keypoint writers) as a small C library (no CUDA)."""
    srcs = [os.path.join(CSRC, f) for f in ("surf_io.cpp", "surf_io.h")] + [os.path.join(ROOT, "include", "frogsurf.h")]
    if not force and _newer(FSIO, srcs):
        return FSIO
    cmd = ["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fopenmp", "-I", os.path.join(ROOT, "include"),
           os.path.join(CSRC, "surf_io.cpp"), "-o", FSIO, "-lz"]
    subprocess.run(cmd, check=True, cwd=ROOT)
    return FSIO


def build_all(force: bool = False) -> None:
    build_lib(force)
    build_cli(force)
    build_fmio(force)
    build_surf_lib(force)
    build_surf_cli(force)
    build_fsio(force)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv)
    print(LIB)
    print(BIN)
