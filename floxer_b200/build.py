"""Builds floxer_b200/libfloxer_gpu.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "csrc", f) for f in ("floxer_gpu.cu", "pex_tree.cpp", "sam_output.cpp", "bam_output.cpp", "seeder.cpp")]
HEADERS = [os.path.join(HERE, "csrc", "bam_kernels.cuh"), os.path.join(HERE, "csrc", "dp_kernels.cuh"), os.path.join(HERE, "csrc", "root_kernels.cuh"), os.path.join(HERE, "csrc", "sam_kernels.cuh"), os.path.join(HERE, "csrc", "seed_kernels.cuh"), os.path.join(os.path.dirname(HERE), "include", "floxer_gpu.h")]
OUTPUT = os.path.join(HERE, "libfloxer_gpu.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-Wall,-Wextra", "-shared"]


def is_stale() -> bool:
    if not os.path.exists(OUTPUT):
        return True
    t = os.path.getmtime(OUTPUT)
    return any(os.path.getmtime(p) > t for p in SOURCES + HEADERS)


def build_native(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return OUTPUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = "nvcc"
    cmd = [nvcc, *NVCC_FLAGS, "-o", OUTPUT, *SOURCES, "-lz"]        # zlib: BGZF blocks of the BAM writer
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        sys.stderr.write(r.stderr)
    return OUTPUT


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose="-v" in sys.argv))
