"""In-tree build of librlfc.so (the C-ABI shared library) with nvcc for sm_100a.

--fmad=false is part of the numerical contract: the reference arithmetic is Java `float` with one
rounding per operation, and the device code must not contract a*b+c into an FMA.
"""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "librlfc.so"
SOURCES = ["rlfc_api.cu", "solver_kernels.cu", "geometry.cpp", "vmm.cpp"]
HEADERS = ["solver.h", "geometry.h", "vmm.h", "smooth_rows.cuh", "smooth_wave.cuh", "smooth_chain.cuh", "smooth_chain3.cuh", "smooth_tiny.cuh", "exact_sum.cuh",
           "exact_sum_kernels.cuh", "snapshot.cuh", "records.cuh", "param_sets.cuh", "geometry_device.cuh", "flow_stats.cuh",
           "../../include/rlfc.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "--fmad=false", "-std=c++17",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-O2",
    "-shared", "-cudart", "shared",
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = [CSRC / s for s in SOURCES] + [(CSRC / h).resolve() for h in HEADERS] + [Path(__file__)]
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return LIB
    cmd = [nvcc_path(), *NVCC_FLAGS, "-o", str(LIB), *[str(CSRC / s) for s in SOURCES]]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd))
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stdout + res.stderr)
    return LIB


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
