"""Build libartp.so (hand-written sm_100a CUDA + the C ABI) in-tree with nvcc."""
from __future__ import annotations

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libartp.so")
# (source, extra flags): the geometric kernels need bit-exact fp32 (no FMA contraction, SURVEY.md section 7);
# the motion-cost network does not.
SOURCES = [("artp_capi.cu", ["-fmad=false", "-Xcompiler", "-fPIC,-ffp-contract=off"]),
           ("artp_cnn.cu", ["-Xcompiler", "-fPIC"])]
HEADERS = ["artp_device.cuh", "artp_kernels.cuh", "artp_sampler.cuh", "artp_tiles.cuh", "artp_basic.cuh", "artp_roadmap.cuh", "artp_cnn.h", os.path.join("..", "..", "include", "artp.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17"]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in [x[0] for x in SOURCES] + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    objs = []
    for src, extra in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, os.path.join(CSRC, src)]
        subprocess.run(cmd, check=True)
        objs.append(obj)
    subprocess.run([nvcc, "-shared", "-o", LIB] + objs, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
