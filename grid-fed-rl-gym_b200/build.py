"""Builds ``libgfr_b200.so`` in-tree with nvcc for sm_100a: ``python -m grid_fed_rl_b200.build``."""

from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libgfr_b200.so")
SOURCES = ["gfr_b200.cu"]
DEPENDS = ["gfr_b200.cu", "gfr_device.cuh", "gfr_dense.cuh", "gfr_image.hpp", os.path.join("..", "..", "include", "gfr_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC", "-cudart", "shared",
              "-Xlinker", "-rpath,/usr/local/cuda/lib64",
              "-Xlinker", "-Bsymbolic"]          # calls between the library's own entry points never leave it


def find_nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: the CUDA toolkit is needed to build libgfr_b200.so")
    return nvcc


def up_to_date() -> bool:
    if not os.path.exists(OUT):
        return False
    t = os.path.getmtime(OUT)
    return all(os.path.getmtime(os.path.join(CSRC, d)) <= t for d in DEPENDS)


STRESS_OUT = os.path.join(HERE, "libgfr_b200_stress.so")


def build_stress(force: bool = False) -> str:
    """The race-hunting twin (-DGFR_STRESS: random delays around every group barrier).  Only
    tests/test_gpu_stress.py loads it, to check that results do not depend on lane timing."""
    if not force and os.path.exists(STRESS_OUT) and all(
            os.path.getmtime(os.path.join(CSRC, d)) <= os.path.getmtime(STRESS_OUT) for d in DEPENDS):
        return STRESS_OUT
    return build(force=True, defines=("GFR_STRESS",), out=STRESS_OUT)


def build(force: bool = False, verbose: bool = False, defines=(), out: str = OUT) -> str:
    if not force and not defines and up_to_date():
        return OUT
    cmd = [find_nvcc(), *NVCC_FLAGS, *[f"-D{d}" for d in defines], "-o", out, *SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        sys.stderr.write(res.stderr)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
