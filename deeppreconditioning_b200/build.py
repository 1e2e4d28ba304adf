"""Build libdpcg.so (hand-written sm_100a CUDA kernels + the C ABI of include/dpcg.h) in-tree with nvcc.

The shared object lands in ``deeppreconditioning_b200/lib/`` (git-ignored, ships to the GPU box with the
snapshot). ``python -m deeppreconditioning_b200.build`` or ``__graft_entry__.build()``.
"""

from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB_DIR = PKG / "lib"
LIB = LIB_DIR / "libdpcg.so"
SOURCES = ["spmv.cu", "scan.cu", "assembly.cu", "levels.cu", "sptrsv.cu", "pcg.cu", "icholt.cu", "sparseconv.cu",
           "sparseconv_grad.cu", "losses.cu", "fsai.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17", "--fmad=false",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "-shared", "--threads", "0",
]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: libdpcg.so cannot be built")


def stale() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "dpcg.h", Path(__file__)]
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False, out: Path = LIB) -> Path:
    """Compile libdpcg.so to ``out`` (default: ``lib/libdpcg.so`` in the package). Without ``force`` nothing is compiled
    while that default library is newer than its sources."""
    if not force and not stale():
        return LIB
    out.parent.mkdir(parents=True, exist_ok=True)
    cmd = [nvcc(), *NVCC_FLAGS, *(["-Xptxas", "-v"] if verbose else []), "-o", str(out), *[str(CSRC / s) for s in SOURCES]]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or proc.returncode:
        sys.stderr.write(proc.stdout + proc.stderr)
    if proc.returncode:
        raise RuntimeError("nvcc failed building libdpcg.so")
    return out


def build_variant(tag: str, defines: dict[str, int]) -> Path:
    """Tuning build: libdpcg_<tag>.so with -D overrides of the pipeline constants (select it with DPCG_LIB)."""
    LIB_DIR.mkdir(exist_ok=True)
    out = LIB_DIR / f"libdpcg_{tag}.so"
    cmd = [nvcc(), *NVCC_FLAGS, *[f"-D{k}={v}" for k, v in defines.items()], "-o", str(out), *[str(CSRC / s) for s in SOURCES]]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode:
        sys.stderr.write(proc.stdout + proc.stderr)
        raise RuntimeError(f"nvcc failed building {out.name}")
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
