"""Build libpmmh_qn_b200.so in-tree with nvcc for sm_100a (B200).

nvcc cross-compiles without a GPU, so this runs in the CPU-only build container as well as
on the GPU box.  The library is written to ``pmmh-qn_b200/lib/`` (git-ignored, but it
travels with the repository snapshot to the GPU box).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libpmmh_qn_b200.so")
SOURCES = ["sv_filter.cu", "sv_fast.cu", "sv_chain.cu", "sv_split.cu", "sv_grid.cu", "aux_kernels.cu", "capi.cu"]
HEADERS = ["common.cuh", "sv_filter.cuh", "sv_math.cuh", "aux_kernels.cuh", "philox.cuh", "sv_split.cuh", "sv_grid.cuh", "sv_call.h", "pf_model.cuh", os.path.join("..", "..", "include", "pmmh_qn.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",            # parity: the reference is plain IEEE fp64 without contraction
    "-Xcompiler", "-fPIC", "-shared",
]


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > built for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    os.makedirs(LIB_DIR, exist_ok=True)
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
        ["-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libpmmh_qn_b200.so")
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
