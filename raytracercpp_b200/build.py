"""Builds raytracercpp_b200/librtb200.so (the C-ABI library: CUDA kernels for sm_100a + host octree builder).

Usage: python -m raytracercpp_b200.build [--force] [--verbose]
nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "librtb200.so"
SOURCES = [CSRC / "rtb200.cu", CSRC / "octree_build.cpp", CSRC / "scene_io.cpp"]
HEADERS = [CSRC / "kernels.cuh", CSRC / "octree_device.cuh", CSRC / "light_cull.cuh", CSRC / "host_common.h", CSRC / "rt_device.h", CSRC / "rt_math.h", CSRC / "scene_layout.h",
           CSRC / "ssao.cuh", CSRC / "ssao_device.h", CSRC / "raster.cuh", CSRC / "raster_device.h",
           PKG.parent / "include" / "rtb200.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    # arithmetic contract of rt_math.h: no FMA contraction, IEEE division and square root
    "--fmad=false", "--prec-div=true", "--prec-sqrt=true",
    "-Xcompiler", "-fPIC,-fopenmp,-ffp-contract=off,-O3",
    "-ccbin", "/usr/bin/g++",
    "-shared", "-lgomp",
]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found")


def up_to_date() -> bool:
    if not LIB.exists():
        return False
    t = LIB.stat().st_mtime
    return all(p.stat().st_mtime <= t for p in SOURCES + HEADERS + [Path(__file__)])


def build(force: bool = False, verbose: bool = False, extra=(), out: Path | None = None) -> Path:
    if out is None and not force and up_to_date():
        return LIB
    cmd = [nvcc(), *NVCC_FLAGS, *extra, "-o", str(out or LIB), *map(str, SOURCES)]
    if verbose:
        print(" ".join(cmd), flush=True)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode:
        raise RuntimeError("nvcc failed")
    return out or LIB


if __name__ == "__main__":
    # extra -D... arguments and --out <file> build a variant of the same sources next to the product library
    argv = sys.argv[1:]
    out = Path(argv[argv.index("--out") + 1]) if "--out" in argv else None
    extra = [a for a in argv if a.startswith("-D")] + (["-Xptxas", "-v"] if "--ptxas" in argv else [])
    print(build(force="--force" in argv, verbose=True, extra=extra, out=out))
