"""Builds the native pieces in-tree (the .so / binaries travel to the GPU box with the snapshot):

  bitmapperbs_b200/libbmbs_gpu.so   CUDA kernels + C ABI (nvcc, sm_100a only)
  bitmapperbs_b200/_build/bmbs       BitMapperBS-compatible command line (host C++ over the C ABI)
  bitmapperbs_b200/_build/bmbs-index index writer (CPU)
  bitmapperbs_b200/_build/bmbs-index-gpu the same files with the suffix sort and the BWT passes on the device (data prep for the 3.1 Gbp bench genome)
"""
from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
OUT = PKG / "_build"
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]
LIB = PKG / "libbmbs_gpu.so"


def _newer(target: Path, sources) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(s).stat().st_mtime > t for s in sources)


def _run(cmd):
    print("+", " ".join(str(c) for c in cmd), file=sys.stderr)
    subprocess.run([str(c) for c in cmd], check=True)


def build_library(force=False) -> Path:
    src = [PKG / "csrc/bmbs_api.cu", PKG / "csrc/bmbs_kernels.cuh", PKG / "csrc/bmbs_device.cuh", PKG / "csrc/bmbs_sort_replay.h", PKG / "csrc/bmbs_band_walk.h", PKG / "csrc/bmbs_refine_ends.h", PKG / "csrc/bmbs_finish_pe.cuh", ROOT / "include/bmbs.h"]
    if force or _newer(LIB, src):
        _run([NVCC, *NVCC_FLAGS, "-shared", src[0], "-o", LIB])
    return LIB


def build_tools(force=False):
    OUT.mkdir(exist_ok=True)
    host = sorted((PKG / "csrc/host").glob("*.hpp")) + sorted((PKG / "indexer").glob("*.hpp")) + [PKG / "csrc/bmbs_refine_ends.h"]
    idx = OUT / "bmbs-index"
    if force or _newer(idx, [PKG / "indexer/build_index.cpp", *host]):
        _run(["g++", "-O2", "-std=c++17", "-pthread", PKG / "indexer/build_index.cpp", "-o", idx])
    gidx = OUT / "bmbs-index-gpu"
    if force or _newer(gidx, [PKG / "indexer/gpu_index.cu", *host]):
        _run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-w", PKG / "indexer/gpu_index.cu", "-o", gidx])
    exe = OUT / "bmbs"
    if force or _newer(exe, [PKG / "csrc/host/bmbs_main.cpp", *host, LIB]):
        _run(["g++", "-O2", "-std=c++17", "-pthread", PKG / "csrc/host/bmbs_main.cpp", "-o", exe,
              f"-L{PKG}", "-lbmbs_gpu", f"-Wl,-rpath,{PKG}", "-Wl,-rpath,$ORIGIN/..", "-lz"])
    return idx, exe


def build_all(force=False):
    build_library(force)
    return build_tools(force)


if __name__ == "__main__":
    build_all("--force" in sys.argv)
