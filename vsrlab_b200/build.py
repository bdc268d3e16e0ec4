"""Build libvsrb200.so in-tree with nvcc for sm_100a:  python -m vsrlab_b200.build"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
SOURCES = ["api.cu", "conv_tc.cu", "conv_ring.cu", "conv_f32.cu", "warp.cu", "train.cu", "wgrad_tc.cu", "wgrad_taps.cu", "loss.cu"]
OUT = CSRC / "libvsrb200.so"
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC", "-shared", "--threads", "0"]      # the six translation units compile in parallel


def needs_build() -> bool:
    if not OUT.exists():
        return True
    t = OUT.stat().st_mtime
    deps = [CSRC / s for s in SOURCES] + [CSRC / "common.cuh", CSRC / "tc_ptx.cuh", CSRC / "warp_modes.cuh", HERE.parent / "include" / "vsrb200.h"]
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return OUT
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).exists():
        raise RuntimeError("nvcc not found: cannot build libvsrb200.so")
    cmd = [nvcc, *FLAGS, "-o", str(OUT), *[str(CSRC / s) for s in SOURCES]]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd))
    subprocess.run(cmd, check=True, cwd=str(CSRC))
    return OUT


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(p)
