"""Builds libporo.so (sm_100a only) in-tree with nvcc; no torch dependency in the library."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libporo.so")
SOURCES = ["vec.cu", "spmv.cu", "stencil.cu", "mg.cu", "bsr.cu", "bsr_tma.cu", "setup.cu", "amg.cu", "distamg.cu", "solver.cu", "sparse_lu.cu", "ilu.cu", "dist.cu", "gen.cu", "capi.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "--extended-lambda",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default", "-Xptxas", "-v" if os.environ.get("PORO_PTXAS_V") else "-O3"]


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "poro.h"))
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            cmd = [NVCC, *FLAGS, "-c", s, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout[-4000:], r.stderr[-8000:]))
            if verbose and r.stderr.strip():
                print(r.stderr)
        return o

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(OUT, objs):
        cmd = [NVCC, "-shared", "-o", OUT, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
