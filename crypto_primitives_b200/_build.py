"""Builds libcpb200.so (hand-written sm_100a CUDA + the C-ABI of include/cpb200.h) in-tree.

nvcc cross-compiles without a GPU; the .so and the objects are git-ignored build products of this
tree.  One translation unit per .cu file, compiled in parallel.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.environ.get("CPB_OBJ_DIR", os.path.join(HERE, "_obj"))     # per tree: a shared directory would hand one checkout another's objects
LIB = os.path.join(HERE, os.environ.get("CPB_LIB_NAME", "libcpb200.so"))
EXTRA = os.environ.get("CPB_NVCC_EXTRA", "").split()
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC",]


def sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _newest_dep() -> float:
    t = 0.0
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for f in os.listdir(root):
            t = max(t, os.path.getmtime(os.path.join(root, f)))
    return t


def needs_build() -> bool:
    return not os.path.exists(LIB) or os.path.getmtime(LIB) < _newest_dep()


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    srcs = sources()
    dep_t = _newest_dep()

    def compile_one(src):
        obj = os.path.join(OBJ, src[:-3] + ".o")
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= dep_t:
            return obj
        cmd = [NVCC, *FLAGS, *EXTRA, "-Xptxas", "-v", "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError(f"nvcc failed on {src}")
        log = os.path.join(OBJ, src[:-3] + ".ptxas.log")
        with open(log, "w") as f:
            f.write(r.stderr)
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    cmd = [NVCC, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static", "-lpthread", "-ldl", "-lrt"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
