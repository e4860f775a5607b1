"""In-tree build of the CUDA library (sm_100a only).  `python -m paillier_halo2_b200.build`.

nvcc cross-compiles without a GPU; the resulting libpaillier_b200.so stays in-tree (git-ignored) so
it travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libpaillier_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC"]
SOURCES = ["capi.cu", "simple64_kernels.cu", "block28_kernels.cu", "cells.cu", "inverse_kernels.cu"]


def _deps_hash(src: str) -> str:
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for name in sorted(os.listdir(root)):
            p = os.path.join(root, name)
            if os.path.isfile(p) and name.endswith((".cu", ".cuh", ".hpp", ".h")):
                if name.endswith(".cu") and name != src:
                    continue
                h.update(name.encode())
                h.update(open(p, "rb").read())
    h.update(" ".join(ARCH + FLAGS).encode())
    return h.hexdigest()


def _compile(src: str, verbose: bool) -> str:
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    stamp = obj + ".hash"
    want = _deps_hash(src)
    if os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == want:
        return obj
    cmd = [NVCC] + ARCH + FLAGS + ["-Xptxas", "-v" if verbose else "-warn-spills", "-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError(f"nvcc failed on {src}")
    if verbose:
        sys.stderr.write(r.stderr)
    open(stamp, "w").write(want)
    return obj


def build(verbose: bool = False, force: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    if force:
        for f in os.listdir(OBJ):
            os.remove(os.path.join(OBJ, f))
    with ThreadPoolExecutor(max_workers=4) as ex:
        objs = list(ex.map(lambda s: _compile(s, verbose), SOURCES))
    newest = max(os.path.getmtime(o) for o in objs)
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < newest:
        cmd = [NVCC] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
