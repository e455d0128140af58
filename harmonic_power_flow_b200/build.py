"""Build the CUDA shared library IN-TREE (harmonic_power_flow_b200/libhpf_b200.so).

Plain nvcc for sm_100a only; no torch headers are involved - the library is a
pure C ABI (include/hpf_b200.h) on top of the CUDA runtime (linked statically,
so it loads on a box without a GPU and fails at hpf_create instead).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libhpf_b200.so")
SOURCES = ["hpf_kernels.cu"]
DEPS = ["hpf_device.cuh", "hpf_zgemm.cuh", "hpf_lu_panel.cuh", "hpf_structured.cuh", "hpf_lane.cuh", "hpf_harmonic_warp.cuh", "hpf_lu_blocked.cuh", "hpf_lockstep.cuh", "hpf_ne_extract.cuh", "hpf_stats.cuh", os.path.join(ROOT, "include", "hpf_b200.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--shared", "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set $NVCC)")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    files = [os.path.join(CSRC, s) for s in SOURCES] + \
            [d if os.path.isabs(d) else os.path.join(CSRC, d) for d in DEPS]
    return any(os.path.getmtime(f) > t for f in files)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    # $HPF_BUILD_FAST=1: ptxas compiles the kernels in parallel (development builds, 3x faster).  NOT for
    # measurements: the split compile allocates registers differently (ls_border_kernel 64 instead of 78,
    # ls_backsub_kernel 40 instead of 32 registers) and those kernels run 15-20 % slower - measured same-box.
    fast = ["--split-compile", "0"] if os.environ.get("HPF_BUILD_FAST") else []
    cmd = [_nvcc()] + NVCC_FLAGS + fast + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed (exit %d): %s" % (r.returncode, " ".join(cmd)))
    with open(os.path.join(PKG, "build_ptxas.log"), "w") as f:
        f.write(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
