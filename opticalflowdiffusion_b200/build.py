"""Builds ``opticalflowdiffusion_b200/lib/libflowdiff.so`` (sm_100a only) with nvcc.

Usage:  python -m opticalflowdiffusion_b200.build [--force] [--verbose]

The library is built in-tree so that it travels to the GPU box with the repository snapshot;
each translation unit is compiled to an object file (cached on its mtime) and linked with
``-cudart shared`` so the library shares the CUDA runtime (and therefore the primary context and
streams) that PyTorch already loaded.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libflowdiff.so")
OBJDIR = os.path.join(LIBDIR, "obj")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr",
    "-DFD_BUILDING_LIB",
]
if os.environ.get("FD_DIAG"):           # diagnostic build: compiles the *_DBG switches into the kernels (fd_common.cuh)
    NVCC_FLAGS.append("-DFD_DIAG")


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _deps_mtime() -> float:
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "flowdiff.h"))
    return max(os.path.getmtime(h) for h in hdrs if os.path.exists(h))


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJDIR, exist_ok=True)
    hdr_m = _deps_mtime()
    objs, jobs = [], []
    for src in sources():
        obj = os.path.join(OBJDIR, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_m):
            cmd = [_nvcc(), *NVCC_FLAGS, "-c", src, "-o", obj]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r.stdout + r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for out in ex.map(run, jobs):
                if verbose and out.strip():
                    print(out)
    if jobs or not os.path.exists(LIB):
        cmd = [_nvcc(), "-shared", "-cudart", "shared", "-gencode", "arch=compute_100a,code=sm_100a",
               "-o", LIB, *objs]
        run(cmd)
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
