"""Build libhymet_screen.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libhymet_screen.so")
SOURCES = ["abi.cu", "screen_kernels.cu", "distance_kernels.cu", "lca_kernels.cu", "msh_capnp.cpp", "fasta_pack.cpp"]
HEADERS = ["kmer_core.cuh", "table_device.cuh", "cuda_owned.h", "screen_kernels.h", "distance_kernels.h", "lca_kernels.h", "msh_capnp.h", "fasta_pack.h",
           os.path.join("..", "..", "include", "hymet_screen.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden,-pthread", "--shared", "-cudart", "shared"]


def stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          [os.path.join(CSRC, f) for f in SOURCES] + ["-o", LIB, "-lz"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libhymet_screen.so")
    if verbose:
        sys.stderr.write(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
