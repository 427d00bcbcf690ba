"""A/B of the small-system Cholesky: prints a hash of dxi and per-phase times for one scene.
Run it from two builds of the library and compare the hashes and the times.

    python tools/chol_ab.py --cams 50 --points 10000
"""
import argparse
import hashlib
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import ba_b200  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--cams", type=int, default=50)
ap.add_argument("--points", type=int, default=10000)
ap.add_argument("--iters", type=int, default=10)
args = ap.parse_args()
sc = ba_b200.scenes.make_scene(args.cams, args.points, seed=1, visibility=1.0)
adj = ba_b200.BundleAdjuster.from_observations(sc.obs_ptr, sc.obs_cam, sc.obs_xy, sc.X0, sc.K0, sc.R0, sc.t0,
                                               f0=sc.f0, axis=sc.axis, dense=sc.dense)
eng = adj.engine
eng.linearize()
eng.build_reduced(1e-4)
eng.solve_trial(1e-4)
dxi = eng.buffer("DXI")
print("dxi sha1", hashlib.sha1(np.ascontiguousarray(dxi).tobytes()).hexdigest(), "norm", float(np.linalg.norm(dxi)))
eng.set_state(adj._X, adj._R, adj._t, adj._f, adj._u)
eng.lm_run(2.0, -1.0, 2)
eng.set_state(adj._X, adj._R, adj._t, adj._f, adj._u)
eng.profile_enable(True)
eng.profile_reset()
recs, st = eng.lm_run(2.0, -1.0, args.iters)
prof = eng.profile()
print(f"{args.cams}x{args.points}: solves={st.solves} E={recs[-1].E:.12g}")
print({k: round(v["ms"] / max(st.solves, 1), 4) for k, v in prof.items()}, "(ms per solve)")
