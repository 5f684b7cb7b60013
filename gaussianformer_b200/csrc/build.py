"""Builds libgf_b200.so (the C-ABI library) in-tree with nvcc for sm_100a.

Run as ``python -m gaussianformer_b200.csrc.build`` or through ``__graft_entry__.build()``.
The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SOURCES = ["cabi.cu", "splat_prep.cu", "splat_forward.cu", "splat_backward.cu", "splat_backward_bin.cu", "daf.cu", "daf_fused.cu", "daf_tma.cu", "occ_loss.cu"]
LIB = os.path.join(HERE, "libgf_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "--expt-relaxed-constexpr",
    "-I", os.path.join(ROOT, "include"), "-I", HERE,
]
# the image exports CC/CXX pointing at a wrapper without a full toolchain; use the system g++
HOST_CXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else None


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(HERE, f) for f in SOURCES + ["common.cuh", "splat_render.cuh", "splat_tile.cuh", "splat_bwd_common.cuh", "daf_pair.cuh"]] + [os.path.join(ROOT, "include", "gf_b200.h"), os.path.join(ROOT, "include", "gf_b200_debug.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, src.replace(".cu", ".o"))
        cmd = [NVCC] + FLAGS + (["-ccbin", HOST_CXX] if HOST_CXX else []) + (["-Xptxas", "-v"] if verbose else []) + [
            "-c", os.path.join(HERE, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {src}\n{out}\n")
        failed = failed or pr.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [NVCC, "-shared", "-o", LIB] + (["-ccbin", HOST_CXX] if HOST_CXX else []) + objs + ["-lcudart"]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
