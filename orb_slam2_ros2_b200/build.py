"""Build liborbx.so (the C-ABI library with the sm_100a kernels) in-tree with nvcc.

    python -m orb_slam2_ros2_b200.build [--force]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "liborbx.so")
SOURCES = ["orbx_kernels.cu", "orbx_match.cu", "orbx_serialize.cu", "orbx_bow.cu", "orbx_vocab.cu", "orbx_bowdb.cu", "orbx_loop.cu", "orbx_sequence.cu", "orbx_api.cu"]
HEADERS = [os.path.join(CSRC, "orbx_device.cuh"), os.path.join(CSRC, "orbx_match.cuh"), os.path.join(CSRC, "orbx_internal.h"), os.path.join(HERE, "..", "include", "orbx.h"), os.path.join(HERE, "..", "include", "orbx_pattern.h")]


def nvcc_cmd(extra=()):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return [
        nvcc,
        "-gencode", "arch=compute_100a,code=sm_100a",
        "-O3", "-lineinfo", "-std=c++17",
        "-ccbin", "/usr/bin/g++",  # the image's CC/CXX=/opt/gcc links libstdc++ statically (dangling symlink)
        "-Xcompiler", "-fPIC,-O2,-Wall",
        "-shared", "-cudart", "static", "--threads", "6",
        *extra,
        "-o", LIB,
        *[os.path.join(CSRC, s) for s in SOURCES],
    ]


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if force or needs_build():
        cmd = nvcc_cmd(("-Xptxas", "-v") if verbose else ())
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
        if verbose:
            sys.stderr.write(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
