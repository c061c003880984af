"""Build libothello_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m subproc_b200.build [--force]

No torch involved: the library is plain CUDA behind ``extern "C"`` (include/othello_b200.h).
The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libothello_b200.so")
SOURCES = ("rules.cu", "playout.cu", "greedy.cu", "perft.cu", "learn.cu", "learn_solve.cu", "value_table.cu", "peak.cu", "host_api.cu",
           "solve.cu", "search.cu", "search_playout.cu", "move_values.cu")
HEADERS = ("bitboard.cuh", "eval.cuh", "fastboard.cuh", "opening_book.cuh", "endgame.cuh", "midgame.cuh", "move_values.cuh", "playout_common.cuh", "common.cuh", os.path.join("..", "..", "include", "othello_b200.h"))

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.isfile(exe):
        raise RuntimeError("nvcc not found; cannot build libothello_b200.so")
    return exe


def stale():
    if not os.path.isfile(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), out=SO):
    """defines / out: experimental variants (tools/ab.sh); the product is the default build"""
    if not force and not defines and out == SO and not stale():
        return SO
    cmd = [nvcc()] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + \
          [os.path.join(CSRC, f) for f in SOURCES]
    subprocess.check_call(cmd)
    return out


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a[2:] for a in sys.argv[1:] if a.startswith("-o")]
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, defines=defs, out=outs[0] if outs else SO))
