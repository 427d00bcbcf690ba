"""Marginal covariances (ba_covariance): time per call and per kernel on the GPU, with the achieved
FP64 rate of the forward substitution against the algorithmic flop counts.

    python tools/time_covariance.py [--out DIR] [--cases c2,c3,s1000] [--reps R]

Flops (algorithmic): point pass 3N n^2 (a triangular solve of 3N rows by L, n = 9M), camera pass
n^3 / 3 (unit rows, leading zeros skipped).  Peak: 37.1 TF/s, the DMMA.8x8x4 rate measured on a B200
(ba_fp64_peak).  Whole-call times are host clocks around a call that ends in a stream
synchronisation, after one warm-up call of the same shape; kernel times come from a separate
torch.profiler run.  Writes r7_covariance_<case>.json into DIR (default profiles/) and, where nvcc
is on the path, r7_covariance_ptxas.txt: the ptxas -v lines of csrc/k8_covariance.cu and the
DMMA.8x8x4 count of each kernel's SASS.
"""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import ba_b200  # noqa: E402
from oracle import ba_oracle as O  # noqa: E402

DMMA_PEAK = 37.1e12
CASES = {"c2": dict(ba_b200.scenes.CONFIGS["c2"]), "c3": dict(ba_b200.scenes.CONFIGS["c3"]),
         "s1000": dict(n_cams=1000, n_points=100_000, seed=7, visibility=0.1)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def ptxas_report(path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        return
    src = os.path.join(ROOT, "3d-reconstruction-from-multi-view-exp_b200", "csrc", "k8_covariance.cu")
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "k8.o")
        res = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v",
                              "-I", os.path.join(ROOT, "include"), "-I", os.path.dirname(src), "-c", src, "-o", obj],
                             capture_output=True, text=True)
        sass = subprocess.run([os.path.join(os.path.dirname(nvcc), "cuobjdump"), "-sass", obj],
                              capture_output=True, text=True).stdout
    counts, cur = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = 0
        elif cur and "DMMA.8x8x4" in line:
            counts[cur] += 1
    version = subprocess.run([nvcc, "--version"], capture_output=True, text=True).stdout.strip().splitlines()[-1]
    with open(path, "w") as fh:
        fh.write(f"# {version}: -O3 -gencode arch=compute_100a,code=sm_100a -Xptxas -v on csrc/k8_covariance.cu\n")
        fh.write("\n".join(l for l in res.stderr.splitlines() if l.strip() and "Compile time" not in l) + "\n\n")
        fh.write("# cuobjdump -sass: DMMA.8x8x4 instructions per kernel (static count)\n")
        fh.writelines(f"{k} {v}\n" for k, v in counts.items())


def engine_for(cfg):
    sc = ba_b200.scenes.make_scene(**cfg)
    X, R, t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, sc.axis)
    eng = ba_b200.Engine(sc.n_points, sc.n_cams, sc.nobs, sc.f0, sc.axis, sc.dense)
    eng.set_observations(sc.obs_ptr, None if sc.dense else sc.obs_cam, sc.obs_xy)
    eng.set_state(X, R, t, sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy())
    return sc, eng


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--cases", default="c2,c3,s1000")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import torch

    ptxas_report(os.path.join(args.out, "r7_covariance_ptxas.txt"))
    gpu = card()
    for name in args.cases.split(","):
        cfg = CASES[name]
        sc, eng = engine_for(cfg)
        N, M = sc.n_points, sc.n_cams
        n = 9 * M
        flops_pts, flops_cam = 3.0 * N * n * n, n ** 3 / 3.0
        eng.covariance()  # warm-up: module load, pool, the factorisation kernels
        calls = {}
        for label, pts in (("cameras_only", False), ("cameras_and_points", True)):
            ts = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                eng.covariance(points=pts)
                ts.append(time.perf_counter() - t0)
            calls[label] = {"ms_min": 1e3 * min(ts), "ms_median": 1e3 * float(np.median(ts))}
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.covariance()
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            if ev.device_type.name == "CUDA":
                kern[ev.key] = {"ms": ev.device_time_total / 1e3, "count": ev.count}
        trsm_ms = sum(v["ms"] for k, v in kern.items() if "cov_trsm_kernel" in k)
        res = {"case": name, "n_cams": M, "n_points": N, "n_obs": int(sc.nobs), "n": n, "gpu": gpu,
               "reps": args.reps, "call": calls,
               "point_pass_flops": flops_pts, "camera_pass_flops": flops_cam,
               "trsm_ms_one_call": trsm_ms,
               "trsm_tflops": (flops_pts + flops_cam) / (trsm_ms * 1e-3) / 1e12 if trsm_ms else None,
               "share_of_dmma_peak": (flops_pts + flops_cam) / (trsm_ms * 1e-3) / DMMA_PEAK if trsm_ms else None,
               "kernels_one_call": dict(sorted(kern.items(), key=lambda kv: -kv[1]["ms"])[:16])}
        print(json.dumps({k: v for k, v in res.items() if k != "kernels_one_call"}), flush=True)
        with open(os.path.join(args.out, f"r7_covariance_{name}.json"), "w") as fh:
            json.dump(res, fh, indent=1)
        eng.close()


if __name__ == "__main__":
    main()
