"""Build libba_b200.so in-tree with nvcc for sm_100a (no torch, no cmake).

    python 3d-reconstruction-from-multi-view-exp_b200/csrc/build.py [--force] [--verbose]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
ROOT = os.path.dirname(PKG)
OUT = os.path.join(PKG, "libba_b200.so")
SOURCES = ["ba_engine.cu", "k1_residual_jacobian.cu", "k2_point_blocks.cu", "k3_schur_syrk.cu", "k3_schur_sparse.cu",
           "k4_cholesky_solve.cu", "k4_cholesky.cu", "k5_project.cu", "fp64_peak.cu", "comm_peer.cu", "k6_gauge.cu", "k7_projective_depth.cu",
           "k8_covariance.cu"]
HEADERS = ["ba_common.cuh", os.path.join(ROOT, "include", "ba_b200.h")]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    cc = nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    hdrs = [h if os.path.isabs(h) else os.path.join(HERE, h) for h in HEADERS]
    flags = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-I", os.path.join(ROOT, "include"),
             "-I", HERE] + ARCH
    if verbose:
        flags += ["-Xptxas", "-v"]

    def compile_one(src: str) -> str:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        srcp = os.path.join(HERE, src)
        if force or _stale(obj, [srcp] + hdrs):
            cmd = [cc] + flags + ["-c", srcp, "-o", obj]
            res = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or res.returncode != 0:
                sys.stderr.write(res.stdout + res.stderr)
            if res.returncode != 0:
                raise RuntimeError(f"nvcc failed on {src}")
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(OUT, objs):
        cmd = [cc, "-shared", "-o", OUT] + objs + ARCH + ["-lcudart"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("link failed")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
