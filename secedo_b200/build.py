"""Builds secedo_b200/libsecedo_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "obj")
LIB = os.path.join(HERE, "libsecedo_b200.so")
SOURCES = ["abi.cu", "scan.cu", "filter.cu", "reads.cu", "scatter.cu", "multilocus.cu", "epilogue.cu", "gemm.cu", "synth.cu", "ingest.cu", "spectral.cu", "eigenvalues.cu", "em.cu", "multi.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
         "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(verbose: bool = False, force: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".hpp"))]
    headers.append(os.path.join(HERE, "..", "include", "secedo_b200.h"))
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]

    def compile_one(src: str):
        s, o = os.path.join(CSRC, src), os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            r = subprocess.run([NVCC] + FLAGS + ["-c", s, "-o", o], capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
            with open(o + ".ptxas.log", "w") as f:
                f.write(r.stderr)
            if verbose:
                sys.stderr.write(r.stderr)
        return o

    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(compile_one, srcs))
    if force or _stale(LIB, objs):
        r = subprocess.run([NVCC, "-shared", "-o", LIB] + objs + ["-lcudart", "-lpthread"], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
