"""Build libsbq.so (the product: CUDA kernels + runtime + C ABI) in-tree with nvcc for sm_100a."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsbq.so")
SOURCES = ["sbq.cu", "sbq_builder.cpp"]
DEPS = ["sbq.cu", "sbq_kernels.cuh", "sbq_grid.cuh", "sbq_grid_tma.cuh", "sbq_grid_dual.cuh", "sbq_bias.cuh", "sbq_weights.cuh", "sbq_multi.cuh", "sbq_synth.cuh", "sbq_rawbuild.cuh", "sbq_bootstrap.cuh", "sbq_gibbs.cuh", "sbq_builder.cpp", os.path.join("..", "..", "include", "sbq.h"),
        os.path.join("..", "..", "include", "sbq_builder.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-cudart", "static"]


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build(force=False, verbose=False):
    if not force and not stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("SBQ_NVCC_EXTRA", "").split()
    cmd = [nvcc, *NVCC_FLAGS, *extra] + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    env = dict(os.environ)
    env.pop("CC", None), env.pop("CXX", None)   # this image exports a static-libstdc++ gcc wrapper; use /usr/bin/g++
    subprocess.check_call(cmd, env=env)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
