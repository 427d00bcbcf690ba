"""Projective-depth iteration: GPU time per iteration next to the CPU restatement.

    python tools/time_depth.py [--method primary|dual] [M N iters]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import ba_b200  # noqa: E402
from oracle import depth_oracle as D  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--method", choices=("primary", "dual"), default="primary")
ap.add_argument("case", nargs="*", type=int, help="M N iters")
args = ap.parse_args()
cases = [tuple(args.case)] if len(args.case) == 3 else [(10, 200, 50), (50, 100_000, 10)]
gpu_fn = getattr(ba_b200, "projective_depth_" + args.method)
cpu_fn = getattr(D, "projective_depth_" + args.method)
for M, N, iters in cases:
    sc = ba_b200.scenes.make_scene(M, N, seed=1, visibility=1.0)
    xd, _ = sc.dense_x()
    x = np.concatenate((xd / sc.f0, np.ones((N, M, 1))), axis=2)
    gpu_fn(x, sc.f0, 0.0, 2)  # warm-up (module load, pool)
    t0 = time.perf_counter()
    z, errs = gpu_fn(x, sc.f0, 0.0, iters)
    t_gpu = (time.perf_counter() - t0) / iters
    n_cpu = min(iters, 3 if N > 10_000 else iters)
    t0 = time.perf_counter()
    zo, eo = cpu_fn(x, sc.f0, 0.0, n_cpu)
    t_cpu = (time.perf_counter() - t0) / n_cpu
    print(json.dumps({"method": args.method, "images": M, "points": N, "iterations": iters,
                      "gpu_ms_per_iteration_e2e": 1e3 * t_gpu,
                      "cpu_port_ms_per_iteration": 1e3 * t_cpu, "cpu_threads": os.cpu_count(),
                      "E_gpu": float(errs[n_cpu - 1]), "E_cpu": eo[-1],
                      "note": "GPU: host arrays in, z out, one host read of E per iteration; CPU: the NumPy "
                              "restatement of oracle/depth_oracle.py"}))
