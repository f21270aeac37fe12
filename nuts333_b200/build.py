"""Builds libnutsb200.so (the C-ABI library of include/nutsb200.h) with nvcc for sm_100a.

In-tree output: nuts333_b200/_lib/libnutsb200.so (git-ignored, travels to the GPU box).
"""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "_lib" / "libnutsb200.so"
SOURCES = [CSRC / "nutsb_lib.cu"]
HEADERS = [CSRC / "nutsb_common.cuh", CSRC / "nutsb_kernels.cuh", CSRC / "nutsb_match.cuh", CSRC / "nutsb_speech.cuh", CSRC / "nutsb_multi.cuh",
           PKG.parent / "include" / "nutsb200.h"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared", "-cudart", "static",
              "--expt-relaxed-constexpr"]


def nvcc_path() -> str:
    cand = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(cand).exists():
        raise RuntimeError("nvcc not found: libnutsb200.so cannot be built (there is no CPU fallback)")
    return cand


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    return any(p.stat().st_mtime > t for p in SOURCES + HEADERS + [Path(__file__)])


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return LIB
    LIB.parent.mkdir(parents=True, exist_ok=True)
    extra = os.environ.get("NUTSB_NVCC_EXTRA", "").split()      # e.g. -DNUTSB_TILE_OPS=256 for A/B runs
    cmd = [nvcc_path(), *NVCC_FLAGS, *extra, "-o", str(LIB), *map(str, SOURCES)]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB


GEN_LIB = PKG / "_lib" / "libnutsgen.so"
GEN_SRC = CSRC / "nutsb_gen.c"


def build_gen(force: bool = False) -> Path:
    """The synthetic input generator (host C, shared by the oracle legs and the GPU driver)."""
    if not force and GEN_LIB.exists() and GEN_LIB.stat().st_mtime >= GEN_SRC.stat().st_mtime:
        return GEN_LIB
    GEN_LIB.parent.mkdir(parents=True, exist_ok=True)
    cc = os.environ.get("CC") or shutil.which("gcc") or "cc"
    r = subprocess.run([cc, "-O2", "-std=c99", "-fPIC", "-shared", "-fvisibility=hidden", "-Wall",
                        "-o", str(GEN_LIB), str(GEN_SRC)], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("gcc failed:\n" + r.stderr)
    return GEN_LIB


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_gen(force="--force" in sys.argv))
