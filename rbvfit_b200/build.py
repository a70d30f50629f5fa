"""Build the CUDA shared library in-tree (rbvfit_b200/csrc/librbvfit_b200.so) with nvcc for sm_100a."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "librbvfit_b200.so")
SOURCES = ["rbv_kernels.cu"]
HEADERS = ["rbv_device.cuh", "rbv_sampler.cuh", "rbv_pt.cuh", "rbv_slice.cuh", "rbv_stream.cuh", "rbv_grad.cuh", "rbv_fisher.cuh", "rbv_lm.cuh", "faddeeva_tables.h", os.path.join("..", "..", "include", "rbvfit_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC", "-cudart", "shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source into the in-tree shared library; returns its path."""
    if not force and not needs_build():
        return LIB_PATH
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
