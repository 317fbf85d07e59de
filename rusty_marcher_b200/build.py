"""Builds librm_b200.so (CUDA kernels + C ABI + host scene builder) in-tree with nvcc for sm_100a.

    python -m rusty_marcher_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librm_b200.so")
SOURCES = ["rm_api.cu", "rm_kernels.cu", "rm_lens.cu", "rm_area.cu", "rm_rough.cu", "rm_motion.cu", "rm_distributed.cu", "rm_indirect.cu", "rm_path.cu", "rm_scene.cpp", "rm_bvh.cpp", "rm_host.cpp"]
HEADERS = ["rm_math.cuh", "rm_trace.cuh", "rm_fast.cuh", "rm_fast_setup.cuh", "rm_sampled.cuh", "rm_bvh.cuh", "rm_scene.h", "rm_kernels.h", "rm_pool.h",
           os.path.join("..", "..", "include", "rm_b200.h"), os.path.join("..", "..", "include", "rm_b200_host.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",                      # FP32 FMAs are written explicitly; FP64 must never fuse
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-Wall",
    "-shared",
]


def nvcc_path():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not stale():
        return LIB
    extra = os.environ.get("RM_NVCC_EXTRA", "").split()         # experiments: e.g. -DRM_K1_MIN_BLOCKS=4
    cmd = [nvcc_path()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + \
          [os.path.join(CSRC, f) for f in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building librm_b200.so")
    if verbose:
        sys.stderr.write(res.stdout + res.stderr)
    return LIB


EXAMPLE_SRC = os.path.join(os.path.dirname(HERE), "examples", "rm_headless.cpp")
EXAMPLE_BIN = os.path.join(os.path.dirname(HERE), "examples", "rm_headless")


def build_examples(force=False):
    """examples/rm_headless: the headless C++ stand-in for the reference's GTK front end, over the C ABI only."""
    build()
    if (not force and os.path.exists(EXAMPLE_BIN)
            and os.path.getmtime(EXAMPLE_BIN) >= max(os.path.getmtime(EXAMPLE_SRC), os.path.getmtime(LIB))):
        return EXAMPLE_BIN
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(os.path.dirname(HERE), "include"), EXAMPLE_SRC, "-o", EXAMPLE_BIN,
           "-L", HERE, "-lrm_b200", "-Wl,-rpath," + HERE]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("g++ failed building examples/rm_headless")
    return EXAMPLE_BIN


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
