"""Build recipe for libkmerml_b200.so (hand-written sm_100a CUDA + the C-ABI).

    python -m kmerml_b200.build [--force] [--verbose]

nvcc cross-compiles for sm_100a without a GPU; the .so is built in-tree (it is
git-ignored but travels to the GPU box with the repo snapshot).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libkmerml_b200.so")
SOURCES = ["api.cu", "dense.cu", "features.cu", "sparse.cu", "sketch.cu", "gram_tc.cu", "format.cu", "hostpipe.cu", "stats.cu", "featcsv.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function",
    "-shared", "-cudart", "static", "-Xcompiler", "-pthread", "-ldl",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return "nvcc"


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(HERE, "..", "include", "kmerml_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else [])
    cmd += ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(LIB)
