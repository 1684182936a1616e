"""Builds llamole_b200/libllamole_b200.so (sm_100a only) with nvcc, in-tree.

    python -m llamole_b200.build [--force]

The library is a plain C-ABI shared object (include/llamole_b200.h); it links the CUDA runtime statically and
resolves the one driver symbol it needs (cuTensorMapEncodeTiled) at run time, so it loads on a machine
without a GPU (symbol checks) and refuses to compute there.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "csrc", "_obj")
LIB = os.path.join(HERE, "libllamole_b200.so")
SOURCES = ["llb_runtime.cu", "llb_rowops.cu", "llb_gemm_ln.cu", "llb_dit.cu", "llb_gin.cu", "llb_gin_grad.cu", "llb_dit_grad.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build llamole_b200's sm_100a kernels)")


def _deps_mtime() -> float:
    paths = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))]
    paths.append(os.path.join(os.path.dirname(HERE), "include", "llamole_b200.h"))
    return max(os.path.getmtime(p) for p in paths)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _deps_mtime():
        return LIB
    nvcc = _nvcc()
    os.makedirs(OBJ, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *os.environ.get("LLB_EXTRA_NVCC_FLAGS", "").split(), "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose and r.stderr:
            print(r.stderr, file=sys.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
