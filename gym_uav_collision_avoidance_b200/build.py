"""In-tree build of libuavca.so (hand-written sm_100a CUDA behind the C-ABI of include/uavca.h)."""
from __future__ import annotations

import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libuavca.so")
SOURCES = ["uavca_kernels.cu", "uavca_policy.cu", "uavca_capi.cu"]
HEADERS = ["uavca_device.cuh", "uavca_multi.cuh", "uavca_seq.cuh", "uavca_cta.cuh", "uavca_tma.cuh", "uavca_host.h",
           os.path.join("..", "..", "include", "uavca.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC"]


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libuavca.so (set NVCC=/path/to/nvcc)")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into gym_uav_collision_avoidance_b200/libuavca.so."""
    if not force and not is_stale():
        return LIB_PATH
    cmd = [find_nvcc(), *NVCC_FLAGS, "-shared", "-o", LIB_PATH, *SOURCES]
    if verbose:
        cmd[1:1] = ["-Xptxas", "-v"]
    subprocess.check_call(cmd, cwd=CSRC)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
