"""Builds the C-ABI library `libsplitp_b200.so` in-tree with nvcc for sm_100a.

    python splitp_b200/build.py [--force]

The .so is git-ignored (history stays source-only) but travels to the GPU box with the gpurun
snapshot.  There is no JIT and no CPU fallback: `splitp_b200._lib` fails loudly when the library is
missing.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(HERE, "libsplitp_b200.so")
OBJ = os.path.join(HERE, "build")
SOURCES = ["pack.cu", "count.cu", "wide.cu", "flatten.cu", "pairs.cu", "gram.cu", "score.cu", "sparse.cu", "marginals.cu", "mi_batch.cu",
           "bootstrap.cu", "agglomerate.cu", "pair_rows.cu", "quartets.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
              "-I", INCLUDE]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the splitp_b200 library cannot be built")


def _deps(src):
    d = [os.path.join(CSRC, src), os.path.join(INCLUDE, "splitp_b200.h")]
    d += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    return d


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link the shared library.  Returns the .so path."""
    nvcc = _nvcc()
    os.makedirs(OBJ, exist_ok=True)
    jobs = []
    objs = []
    for src in SOURCES:
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, _deps(src)):
            jobs.append([nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj])

    def run(cmd):
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed: {' '.join(cmd)}\n{r.stdout}\n{r.stderr}")
        return r

    with ThreadPoolExecutor(max_workers=min(6, max(1, len(jobs)))) as ex:
        list(ex.map(run, jobs))
    if force or jobs or _stale(LIB, objs):
        run([nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
