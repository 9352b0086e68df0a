"""Build recipe for the in-tree CUDA library (sm_100a only).

`nvcc` cross-compiles without a GPU, so this runs in the CPU build container as
well as on the B200 box.  The resulting `libkirag_b200.so` lives next to this
file: it is git-ignored but travels to the GPU box with the snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libkirag_b200.so")
SOURCES = ["api.cu", "convert.cu", "scan_exact.cu", "rescore.cu", "select.cu", "pool.cu", "scan_tc.cu", "exchange.cu", "range.cu", "multi.cu", "compact.cu"]
HEADERS = ["common.cuh", os.path.join("..", "..", "include", "kirag_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC or put /usr/local/cuda/bin on PATH)")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.join(CSRC, h) for h in HEADERS]
    return any(os.path.getmtime(p) > built for p in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu into libkirag_b200.so; returns the library path."""
    if not force and not is_stale():
        return LIB_PATH
    cmd = [find_nvcc()] + NVCC_FLAGS + ["-o", LIB_PATH] + SOURCES
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    proc = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
        raise RuntimeError(f"nvcc failed with exit code {proc.returncode}")
    if verbose:
        sys.stderr.write(proc.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
