"""Build libhrb200.so (sm_100a only) in-tree with nvcc.  No GPU is needed to build.

    python -m handyrec_b200.build            # incremental
    python -m handyrec_b200.build --force
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libhrb200.so")
SOURCES = ["common.cu", "lookup.cu", "embedding_bwd.cu", "fm.cu", "dense.cu", "gemm_tc.cu", "misc.cu", "lau.cu", "layers_misc.cu", "host_pack.cu", "retrieval.cu", "search.cu", "metrics.cu", "clip.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden",
    "--expt-relaxed-constexpr",
]
if os.environ.get("HRB_DEVTOOLS"):  # perf-debugging hooks (ablation bits, clock64 traces); never set for the shipped library
    FLAGS.append("-DHRB_DEVTOOLS")


def _deps():
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(HERE, "..", "include", "hrb200.h"))
    return hdrs


def _stale(target: str, srcs) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in srcs)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    deps = _deps()
    jobs = []
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + deps):
            jobs.append([NVCC, *FLAGS, "-c", s, "-o", o])

    def run(cmd):
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            list(ex.map(run, jobs))
    if jobs or force or _stale(LIB, objs):
        run([NVCC, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
