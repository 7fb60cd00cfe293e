"""Builds libcfb.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python conformer-nemo_b200/build.py [--force]

nvcc cross-compiles without a GPU.  The .so lands in conformer-nemo_b200/lib/ and travels to the GPU box with the
repository snapshot (it is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
OBJ_DIR = os.path.join(HERE, "build")
LIB_PATH = os.path.join(LIB_DIR, "libcfb.so")

SOURCES = ["engine.cu", "tmap.cu", "gemm_tc.cu", "gemm_tc2.cu", "gemm_simt.cu", "elementwise.cu", "packed.cu", "conv_tail.cu", "attention_tc.cu", "attention_tcp.cu",
           "attention_tc128.cu", "attention_simt.cu", "ctc_head.cu", "frontend.cu", "buffered.cu", "rnnt_greedy.cu",
           "rnnt_beam.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIB_DIR, exist_ok=True)
    os.makedirs(OBJ_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "cfb.h"))
    nvcc = _nvcc()
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ_DIR, src[:-3] + ".o")
        if force or _stale(o, [s] + headers):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc] + NVCC_FLAGS + ["-c", s, "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = r.stdout + r.stderr
        with open(o[:-2] + ".log", "w") as f:
            f.write(log)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {s}:\n{log[-6000:]}")
        return s, log

    if jobs:
        with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for s, log in ex.map(compile_one, jobs):
                if verbose:
                    print(f"== {os.path.basename(s)}\n{log}")
    objs = [os.path.join(OBJ_DIR, src[:-3] + ".o") for src in SOURCES]
    if force or jobs or _stale(LIB_PATH, objs):
        cmd = [nvcc, "-shared", "-o", LIB_PATH] + objs + ["-cudart", "static", "-gencode",
                                                          "arch=compute_100a,code=sm_100a"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return LIB_PATH


if __name__ == "__main__":
    path = build_library(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
