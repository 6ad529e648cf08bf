"""Builds libcalfkit_b200.so in-tree for sm_100a (nvcc cross-compiles without a GPU).

    python calfkit-sdk_b200/build.py [--verbose]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libcalfkit_b200.so")
SRCS = [os.path.join(HERE, "csrc", "ck_api.cu")]
DEPS = SRCS + [os.path.join(HERE, "csrc", f) for f in ("ck_kernels.cuh", "ck_walk.cuh", "ck_float.cuh", "ck_canon.cuh", "ck_plan2.cuh", "ck_gate.cuh", "ck_kafka.cuh", "ck_inflate.cuh", "ck_lz4.cuh", "ck_lz4_enc.cuh", "ck_deflate.cuh", "ck_group.cuh", "ck_xsend.cuh", "ck_fanout2.cuh", "ck_walk_long.cuh", "ck_common.h")] + \
    [os.path.join(HERE, "..", "include", "calfkit_b200.h")]


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and os.path.exists(LIB) and all(os.path.getmtime(d) <= os.path.getmtime(LIB) for d in DEPS):
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "-Xcompiler", "-fPIC,-Wno-stringop-overflow", "-shared", "-o", LIB] + SRCS
    if verbose:
        cmd += ["-Xptxas", "-v"]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose="--verbose" in sys.argv))
