"""Builds the engine's shared library in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m leaf_b200.build          # -> leaf_b200/lib/libleaf_b200.so
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libleaf_b200.so")
SOURCES = ["engine.cu"]
HEADERS = ["gemm_sm100.cuh", "gemm2_sm100.cuh", "train_kernels.cuh", "tower_kernels.cuh", "k1_core.cuh", "k1_tokenize.cuh", "constrain_core.cuh", "constrain_kernel.cuh", "k1_tables_host.h", "k1_tables.inc",
           os.path.join("..", "..", "include", "leaf_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
