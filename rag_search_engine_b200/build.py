"""Build librse.so (the C-ABI CUDA library) in-tree for sm_100a.

    python -m rag_search_engine_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU
box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = CSRC / "librse.so"
SOURCES = [CSRC / "rse.cu"]
HEADERS = sorted(CSRC.glob("*.cuh")) + sorted(CSRC.glob("*.h")) + [PKG.parent / "include" / "rse.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "--fmad=false",                 # no implicit contraction anywhere: parity arithmetic is explicit
    "-Xcompiler", "-fPIC", "-shared",
    "-Xptxas", "-v",
]


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    return any(p.stat().st_mtime > t for p in SOURCES + HEADERS + [Path(__file__)])


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return LIB
    # RSE_EXTRA_NVCC_FLAGS: e.g. -DRSE_REFINE_TIMING for the per-phase stamps scripts/refine_timing.py reads
    extra = os.environ.get("RSE_EXTRA_NVCC_FLAGS", "").split()
    cmd = ["nvcc", *NVCC_FLAGS, *extra, "-o", str(LIB), *map(str, SOURCES)]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    # the log (register / spill counts per kernel) is a build product, kept beside the library and out of git;
    # drop the lines that differ on every build
    log = "\n".join(l for l in (proc.stdout + proc.stderr).splitlines() if "Compile time" not in l) + "\n"
    (CSRC / "build.log").write_text(log)
    if proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
        raise RuntimeError("nvcc failed building librse.so")
    if verbose:
        print(proc.stdout + proc.stderr)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(LIB)
