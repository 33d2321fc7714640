"""Builds libidqn_b200.so (sm_100a only) in-tree with nvcc.  No JIT cache: the .so travels with the repo."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libidqn_b200.so")
SOURCES = ["net.cu", "sumtree.cu", "replay.cu", "peer.cu", "checkpoint.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libidqn_b200.so cannot be built")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(PKG), "include", "idqn_b200.h"))
    objs, jobs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(CSRC, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            jobs.append([nvcc, *NVCC_FLAGS, "-c", s, "-o", o])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
            for log in ex.map(run, jobs):
                if verbose:
                    sys.stderr.write(log)
    if jobs or force or _stale(LIB, objs):
        run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-lcudart"])
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
