"""In-tree build of libtxh.so (hand-written CUDA for sm_100a + the C ABI of include/txh.h).

    python -m tx_fast_hydrology_b200.build [--force]

The shared library is written next to this file so it travels with the repo
snapshot to the GPU box; it is git-ignored (history stays source-only).
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtxh.so")
SOURCES = ["txh_topology.cpp", "txh_geojson.cpp", "txh_route.cu", "txh_window.cu", "txh_lane.cu", "txh_da.cu", "txh_kf.cu", "txh_capi.cu"]
HEADERS = ["txh_topology.hpp", "txh_kernels.cuh", "txh_device.cuh", os.path.join("..", "..", "include", "txh.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-O3",
]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libtxh.so cannot be built (there is no CPU fallback)")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    deps += [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build_lib(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    flags = list(NVCC_FLAGS)
    cmd = [_nvcc()] + flags + ["-shared", "-o", LIB] + srcs + ["-lcudart"]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd))
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)      # the image exports a gcc without OpenMP specs
    subprocess.run(cmd, check=True, env=env)
    return LIB


if __name__ == "__main__":
    build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)
