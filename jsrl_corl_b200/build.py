"""Builds the CUDA engine in-tree: jsrl_corl_b200/libiql_b200.so (sm_100a only).

    python -m jsrl_corl_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the
GPU box with the repo snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libiql_b200.so")
SOURCES = ["engine.cu", "kernels_simt.cu", "kernels_skinny.cu", "replay.cu", "umma_gemm.cu", "fused_fwd.cu", "bwd_chain.cu", "mt19937.cu"]
HEADERS = ["engine.h", "common.cuh", "umma_gemm.h", "tcgen05.cuh", "adam.cuh", os.path.join("..", "..", "include", "iql_b200.h")]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT] + [os.path.join(CSRC, s) for s in SOURCES]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + proc.stdout + proc.stderr)
    if verbose:
        print(proc.stdout + proc.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
