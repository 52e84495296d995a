"""Build the sm_100a CUDA library (limbo_b200/lib/liblimbo_b200.so) in-tree with nvcc.

The library is plain CUDA runtime + C ABI (include/limbo_b200.h); it does not
link against torch.  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "liblimbo_b200.so")
SOURCES = ["abi.cu", "pool.cu", "kbuild.cu", "potrf.cu", "trsv.cu", "query.cu", "query_i8.cu", "lml.cu", "loo.cu", "tf32_query.cu", "sparsify.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "--extended-lambda", "-Xcompiler", "-fPIC", "-diag-suppress", "177",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stamp() -> str:
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for dirpath, _, files in sorted(os.walk(root)):
            for f in sorted(files):
                if f.endswith((".cu", ".cuh", ".h", ".hpp")):
                    with open(os.path.join(dirpath, f), "rb") as fh:
                        h.update(f.encode())
                        h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    stamp_file = os.path.join(LIBDIR, "build.stamp")
    stamp = _stamp()
    if not force and os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(LIBDIR, "obj")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src: str) -> str:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose and (r.stdout or r.stderr):
            print(r.stdout, r.stderr, file=sys.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 2)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp_file, "w") as fh:
        fh.write(stamp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
