"""Build libb200_tetris_mcts.so in-tree with nvcc for sm_100a (no JIT cache: the .so must travel with the repo)."""
import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libb200_tetris_mcts.so")
SOURCES = ["capi.cu", "trainer.cu"]
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC", "-shared"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = ([os.path.join(CSRC, f) for f in SOURCES] + glob.glob(os.path.join(CSRC, "*.cuh"))
            + [os.path.join(HERE, "..", "include", "b200_tetris_mcts.h")])
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, out=None):
    """out: development aid — build the library to another path (e.g. from another checkout, for an A/B comparison); that
    build is loaded instead when the environment names it in B200_TETRIS_LIB (tetris_mcts_b200/_lib.py)."""
    if out is None and not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = "nvcc"
    cmd = [nvcc] + FLAGS + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", out or LIB, "-lcuda"]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd), flush=True)
    subprocess.run(cmd, check=True)
    return out or LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print(LIB)
