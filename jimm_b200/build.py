"""Build libjimm_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m jimm_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The shared object lands next to this file (git-ignored, but it
travels to the GPU box with the snapshot).  cudart is linked statically, cuTensorMapEncodeTiled is
resolved at run time through cudaGetDriverEntryPoint, so the library depends on nothing but libcuda.
"""

from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libjimm_b200.so")
SOURCES = ["gemm.cu", "attention.cu", "attention_tc.cu", "attention_tc_long.cu", "elementwise.cu", "pack.cu", "comm.cu", "preprocess.cu", "postprocess.cu", "probe.cu", "model.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr",
]


def _newest_dep() -> float:
    t = 0.0
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for f in os.listdir(root):
            t = max(t, os.path.getmtime(os.path.join(root, f)))
    return max(t, os.path.getmtime(__file__))


def _stale() -> bool:
    return not os.path.exists(LIB) or os.path.getmtime(LIB) < _newest_dep()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    if not force and not _stale():
        return LIB
    # one builder at a time: under torchrun every rank calls build(); without the lock their nvcc runs overwrite each other's objects and
    # a rank can dlopen a half-written library.  Whoever gets the lock second finds the library fresh and returns.
    import fcntl

    with open(os.path.join(OBJ, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale():
                return LIB
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose: bool) -> str:
    def compile_one(src: str) -> str:
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    tmp = LIB + f".tmp{os.getpid()}"
    cmd = [NVCC, "-shared", "-o", tmp, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, LIB)  # atomic: a concurrent dlopen sees the old or the new library, never a partial one
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
