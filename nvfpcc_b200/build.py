"""In-tree build of the CUDA library (nvcc, sm_100a only).

    python -m nvfpcc_b200.build [--force]

Produces nvfpcc_b200/libnvf_b200.so next to this file.  nvcc cross-compiles
without a GPU, so this also runs in the CPU-only build container.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libnvf_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]           # IEEE arithmetic: --use_fast_math is never passed
UNITS = ("nvf_capi.cu", "nvf_prep.cu", "nvf_entropy.cpp")       # translation units of the one shared library
OBJ_DIR = os.path.join(HERE, "build")


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found")


def sources():
    deps = [os.path.join(ROOT, "include", "nvf_b200.h")]
    deps += [os.path.join(ROOT, "include", "nvf_prep_b200.h")]
    deps += [os.path.join(ROOT, "include", "nvf_metrics_b200.h")]
    deps += [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".h", ".cu", ".cuh", ".cpp", ".inl"))]
    return deps


def stale() -> bool:
    if not os.path.isfile(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(s) > t for s in sources())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return OUT
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()
    extra = ["-Xptxas", "-v"] if verbose else []

    def compile_unit(name: str) -> str:
        obj = os.path.join(OBJ_DIR, os.path.splitext(name)[0] + ".o")
        subprocess.check_call([nvcc] + NVCC_FLAGS + extra + ["-c", "-o", obj, os.path.join(CSRC, name)])
        return obj

    with ThreadPoolExecutor(len(UNITS)) as ex:
        objs = list(ex.map(compile_unit, UNITS))
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", OUT] + objs)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
