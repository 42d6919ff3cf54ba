"""Build libbmf_b200.so (the C-ABI library of include/pybmf_b200.h) in-tree with nvcc for sm_100a.

    python -m pybmf_b200.build            # rebuild if sources are newer than the .so
    python -m pybmf_b200.build --force

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbmf_b200.so")
SOURCES = ["bmf_core.cu", "bmf_bits.cu", "bmf_tc.cu", "bmf_concept.cu"]
HEADERS = [os.path.join(CSRC, "bmf_common.cuh"), os.path.join(HERE, "..", "include", "pybmf_b200.h")]
NVCC_FLAGS = os.environ.get("BMF_EXTRA_NVCC", "").split() + ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libbmf_b200.so cannot be built")


def stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return LIB
    nvcc = nvcc_path()
    objs = []
    for s in SOURCES:
        obj = os.path.join(CSRC, s.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, s), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        subprocess.run(cmd, check=True)
        objs.append(obj)
    subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", *objs, "-o", LIB], check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
