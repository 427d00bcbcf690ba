"""Time the dense Schur product (K3) alone on one scene: the "syrk" profile group, i.e. the DMMA
kernels (syrk_tma_kernel for 128-tiles, syrk_dmma_kernel for 64-tiles) and syrk_reduce_kernel, or
the INT8 emulation's kernels when the engine picks it.

    python tools/syrk_sweep.py --cams 200 --points 100000 [--reps 5]

Prints the SYRK kernel's average launch time, the algorithmic TFLOP/s (3 N n (n + 1), n = 9 M - 7)
and its fraction of the DMMA peak measured on the same GPU.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import ba_b200  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--cams", type=int, default=200)
ap.add_argument("--points", type=int, default=100000)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--tag", default="")
args = ap.parse_args()

N, M = args.points, args.cams
rs = np.random.RandomState(0)
sc = ba_b200.scenes.make_scene(M, min(N, 2000), seed=1)  # cameras + a few points; the rest are drawn cheaply
X = rs.uniform(-1, 1, (N, 3))
f, u = np.ones(M), np.zeros((M, 2))
pt, cam = np.repeat(np.arange(N), M), np.tile(np.arange(M), N)
xy = ba_b200.scenes.project_obs(X, f, u, sc.R_gt, sc.t_gt, 1.0, pt, cam) + 0.005 * rs.standard_normal((N * M, 2))
eng = ba_b200.Engine(N, M, N * M, 1.0, sc.axis, True)
eng.set_observations(None, None, xy)
Xn, Rn, tn = ba_b200.submodule("gauge").normalize(X + 0.01 * rs.standard_normal(X.shape), sc.R0, sc.t0, sc.axis)
eng.set_state(Xn, Rn, tn, 1.05 * f, u)
eng.linearize()
eng.build_reduced(1e-4)  # warm-up
eng.profile_enable(True)
eng.profile_reset()
for k in range(args.reps):
    eng.build_reduced(1e-4 * (k + 2))
prof = eng.profile()
n = 9 * M - 7
flops = 3.0 * N * n * (n + 1.0)
ms = prof["syrk"]["ms"] / prof["syrk"]["launches"]
peak = ba_b200.submodule("engine").fp64_peak(0, True)
print(json.dumps({"tag": args.tag, "cams": M, "points": N, "n_pad": eng.n_pad, "syrk_ms": ms,
                  "k3_ms": prof["k3"]["ms"] / args.reps, "k2_ms": prof["k2"]["ms"] / args.reps,
                  "tflops": flops / ms / 1e9, "peak": peak, "feed": ba_b200.submodule("engine").syrk_feed(), "frac": flops / ms / 1e9 / peak,
                  "env": {k: v for k, v in os.environ.items() if k.startswith("BA_")}}))
