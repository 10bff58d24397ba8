"""Build libjuqbox_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m juqbox_b200.build [--force]

The .so lands in juqbox_b200/lib/ (git-ignored, but it travels to the GPU box with gpurun).
"""
from __future__ import annotations

import glob
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libjuqbox_b200.so")
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "--threads", "0", "-diag-suppress=550,177"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; juqbox_b200 has no CPU fallback and cannot be used without its CUDA library")


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = (sources() + glob.glob(os.path.join(CSRC, "*.h")) + glob.glob(os.path.join(CSRC, "*.cuh")) +
            glob.glob(os.path.join(HERE, "..", "include", "*.h")))
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False, extra_flags=()) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    objs, cmds = [], []
    nvcc = _nvcc()
    hdrs = (glob.glob(os.path.join(CSRC, "*.h")) + glob.glob(os.path.join(CSRC, "*.cuh")) +
            glob.glob(os.path.join(HERE, "..", "include", "*.h")))
    for src in sources():
        obj = os.path.join(LIBDIR, os.path.basename(src)[:-3] + ".o")
        if force or not os.path.exists(obj) or any(os.path.getmtime(d) > os.path.getmtime(obj) for d in [src] + hdrs):
            cmd = [nvcc, *NVCC_FLAGS, *extra_flags, "-c", src, "-o", obj]
            if os.environ.get("JQ_FAST_BUILD"):      # development only: faster, slightly different register allocation
                cmd.insert(1, "--split-compile=0")
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
                print(" ".join(cmd))
            cmds.append(cmd)
        objs.append(obj)
    # the translation units are independent (the trajectory-kernel instantiations are split over jq_traj.cu and jq_traj_inst_*.cu): compile in parallel
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=max(1, min(len(cmds), os.cpu_count() or 1))) as pool:
        list(pool.map(subprocess.check_call, cmds))
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
