"""Build librs_engine.so (the C-ABI library of sm_100a kernels) in-tree with nvcc.

nvcc cross-compiles without a GPU.  Objects are cached under reazonspeech_b200/csrc/build/
and rebuilt when the source (or any header) is newer.  Usage: ``python -m reazonspeech_b200.build``.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "librs_engine.so")
SOURCES = ["gemm_tcgen05.cu", "logmel.cu", "subsample.cu", "elementwise.cu", "resample.cu", "attention_tc.cu", "decode_spec.cu", "decode_alsd.cu", "align.cu", "host_staging.cu", "engine.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
FLAGS += os.environ.get("RS_BUILD_FLAGS", "").split()        # build-time only, e.g. -DRS_PROF for scripts/diag_gemm_timeline.py


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _headers_mtime() -> float:
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hs.append(os.path.join(HERE, "..", "include", "rs_engine.h"))
    return max(os.path.getmtime(h) for h in hs)


def build(force: bool = False, verbose: bool = False) -> str:
    obj_dir, lib = OBJ, LIB
    os.makedirs(obj_dir, exist_ok=True)
    nvcc = _nvcc()
    hm = _headers_mtime()
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(obj_dir, src.replace(".cu", ".o"))
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), hm):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc, *ARCH, *FLAGS, "-c", s, "-o", o]
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {s}:\n{r.stdout}\n{r.stderr}")
        return o

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            list(ex.map(compile_one, jobs))
    objs = [os.path.join(obj_dir, s.replace(".cu", ".o")) for s in SOURCES]
    if jobs or not os.path.exists(lib):
        cmd = [nvcc, *ARCH, "-shared", "-o", lib, *objs]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
