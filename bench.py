#!/usr/bin/env python
"""Benchmark of the bundle-adjustment hot path (BASELINE.json metric: observations/s of
Levenberg-Marquardt iterations, i.e. visible observations x accepted LM iterations / second).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c4|c5] [--weak]
                    [--extras auto|none|c2,c4,c5] [--impl reference] [--dump-outputs DIR]

Headline workload: BASELINE.json config 3 (200 cameras x 100 000 points, full visibility -- the
dense Schur SYRK), one GPU at N = 1 and STRONG-scaled at N > 1: every rank generates its shard of
the same global scene (chunk-seeded generator), the ranks sum the partial reduced system and the
trial cost once per inner solve.  One "step" = one accepted LM iteration (linearise, damped Schur
solve(s), trial cost, accept), started from the same perturbed-ground-truth state every time.

`value`    device-resident: inputs already in HBM, CUDA events around exactly K iterations.
`e2e`      through the reference's own constructor signature with ordinary (pageable) NumPy arrays:
           BundleAdjuster(x (N, M, 2) as np.stack(x_list).transpose(1, 0, 2), X, K, R, t, axis=...)
           .optimize(...) -- H2D of the observations and the state, host gauge passes, K iterations,
           D2H of the result, wall clock; `e2e.from_observations` is the same through the
           observation-list constructor with pinned buffers and the gauge on the device.
`roofline` the dominant kernel (K3, the FP64-tensor-core SYRK): algorithmic flops / launch over its
           CUDA-event duration, against the DMMA peak measured live on this GPU.
`cpu_baseline` the UNMODIFIED reference (oracle/_ref, a build-time copy) on a bounded sample of the
           workload, next to the CPU oracle port on a larger sample.
`parity_vs_n1` (N > 1) the sharded run's per-iteration costs against a single-GPU run of the same
           global scene made in the same invocation (rank 0, scene gathered over NCCL); the bench
           exits non-zero if they differ by more than 1e-9 relative.
`extra`    N = 1: config 2 (50 x 10k, the small latency-bound case) with its own roofline / e2e;
           N = 8: config 4 (1000 cameras x 1M points, 10 % visibility) strong-scaled with parity and
           the sparsity-aware CPU denominator, and config 5 (1 % outliers) run to convergence.

`--dump-outputs DIR` writes the headline's results after its timed steps (see dump_outputs).  The
scenes come from fixed seeds, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "BA LM observations/s (visible observations x accepted LM iterations per second)"
UNIT = "observations/s"
SCALE, TOL_NEVER = 2.0, -1.0  # optimize(2.0, ...) as in the reference script; tol<0: never stop early
PARITY_RTOL = 1e-9

E2E_REPS = 3
CHUNK = 10  # LM iterations per run from the perturbed start (see run_iters)
# bounded CPU samples: points of the named scene (cameras unchanged).  REF_* for the unmodified
# reference ((N, n, n) float64 temporary: 1.6 MB / 25.7 MB / 647 MB per point), PORT_* for the port
# c4 / c5: no sample -- at 10 % visibility every camera needs some hundred points before it is seen at
# all (an unseen camera makes the reference's reduced system singular, :146), and 100 points are 65 GB
REF_SAMPLE = {"c2": 1_000, "c3": 60, "c4": None, "c5": None}
PORT_SAMPLE = {"c2": (10_000, 2), "c3": (1_500, 1), "c4": (20_000, 1), "c5": (20_000, 1)}
DUMP_MAX_BYTES = 64 << 20
DUMP_SEED = 0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "collective"],
                    help="N > 1: how the ranks sum the partial reduced system and the cost: the library's "
                         "own kernels over NVLink peer memory (auto/peer) or torch.distributed all-reduces")
    ap.add_argument("--profile-ranks", action="store_true",
                    help="N > 1: re-run the K iterations with per-phase CUDA-event timing on every rank "
                         "(eager launches) and add rank 0's phase table; `comm` includes waiting for peers")
    ap.add_argument("--weak", action="store_true",
                    help="weak scaling: every rank owns a full named scene of its own (default at N > 1: "
                         "strong, the named scene's points are split over the ranks)")
    ap.add_argument("--strong", action="store_true", help="(default; kept for older command lines)")
    ap.add_argument("--extras", default="auto",
                    help="auto: c2 at N = 1, c4 + c5 at N = 8; none; or a comma list of c2,c4,c5")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the single-GPU parity run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the headline workload's last step computed "
                         "(X, K, R, t in the caller's frame and the costs of the last LM run) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the CUDA arm's outputs")
    return args


def workload_config(name: str) -> dict:
    import ba_b200

    return dict(ba_b200.scenes.CONFIGS[name])


def describe(name: str, cfg: dict, world: int, strong: bool) -> dict:
    vis = cfg.get("visibility", 1.0)
    n_total = cfg["n_points"] if (strong or world == 1) else cfg["n_points"] * world
    d = {
        "workload": f"{name}: synthetic {cfg['n_cams']} cameras x {cfg['n_points']} points"
                    + ("" if (strong or world == 1) else " per GPU")
                    + f", {'full' if vis >= 1.0 else f'{vis:.0%} random'} visibility"
                    + (f", {cfg['outlier_frac']:.0%} outliers" if cfg.get("outlier_frac") else ""),
        "n_cams": cfg["n_cams"], "n_points": n_total,
        "unknowns_reduced": 9 * cfg["n_cams"] - 7,
        "lm": "optimize(scale_factor=2.0), one step = one accepted LM iteration; K steps = LM runs of <= 10 "
              "iterations from the perturbed start (the state is reset on the device between runs)",
        "l2": "no flush: iterations are data-dependent; per-iteration working set "
              "(Jacobian rows + Y) exceeds the 126 MB L2 for c2 and larger",
    }
    if world > 1:
        d["parallelism"] = (f"points {'split' if strong else 'sharded (one named scene per GPU)'} over {world} GPUs, "
                            "cameras replicated")
    else:
        d["parallelism"] = "single GPU"
    return d


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the GPU is under load."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        threading.Thread(target=self._pump, daemon=True).start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        rows = [r for ts, r in self.rows if len(r) >= 8 and (t0 is None or t0 <= ts <= t1)]
        if len(rows) < 3:
            rows = [r for _, r in self.rows if len(r) >= 8]
        sm, reasons, smax = [], set(), None
        for r in rows:
            try:
                sm.append(float(r[1]))
                smax = float(r[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU legs
# ------------------------------------------------------------------------------------------------
def use_all_host_threads() -> int:
    """torchrun exports OMP_NUM_THREADS=1 to its ranks; the CPU legs are meant to use the box's
    host cores, so the BLAS / OpenMP pools are opened up again at run time."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    os.environ["OMP_NUM_THREADS"] = str(n)
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=n)
    except Exception:
        pass
    try:
        import ctypes

        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(n)
    except Exception:
        pass
    return n


def blas_threads() -> int:
    try:
        from threadpoolctl import threadpool_info

        return max([d.get("num_threads", 1) for d in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count() or 1


def sample_scene(name: str, n_points: int):
    import ba_b200

    cfg = workload_config(name)
    cfg["n_points"] = min(n_points, cfg["n_points"])
    return ba_b200.scenes.make_scene(**cfg)


def oracle_port_run(name: str, n_points: int, iters: int):
    """`iters` LM iterations of the CPU oracle port on the first `n_points` points of the workload:
    sparsity-aware C restatement of the Schur reduction + Cholesky for the sparse (1000-camera)
    workloads, the dense GEMM form + LU for the dense ones."""
    from oracle import ba_oracle as O

    sc = sample_scene(name, n_points)
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr)),
                    sc.obs_cam.astype(np.int64), sc.obs_xy, sc.obs_ptr)
    ora = O.OracleBundleAdjuster(None, sc.X0, sc.K0, sc.R0, sc.t0, f0=sc.f0, axis=sc.axis, obs=obs)
    chunk = max(64, min(4096, int(2.5e8 // (27 * sc.n_cams * 8))))
    kw = dict(schur="sparse", solver="cholesky") if not sc.dense else dict(chunk_points=chunk)
    t0 = time.perf_counter()
    ora.optimize(SCALE, TOL_NEVER, max_iter=iters, verbose=False, **kw)
    dt = time.perf_counter() - t0
    done = len(ora.trace) - 1
    solves = sum(r["solves"] for r in ora.trace)
    return {"value": sc.nobs * done / dt, "seconds": dt, "observations": sc.nobs, "iterations": done,
            "solves": solves, "points": sc.n_points, "rms": float(np.sqrt(ora.trace[-1]["E"] / sc.nobs)),
            "formulation": "observation list; " + ("sparsity-aware Schur reduction in C/OpenMP (sum_j 3 (9 m_j)(9 m_j + 1) "
                           "flops), LAPACK Cholesky" if not sc.dense else "dense Schur product as BLAS GEMM per point chunk, LAPACK LU")}


def reference_run(name: str, n_points: int, calls):
    """The UNMODIFIED reference class (oracle/_ref copy of lib/bundle_adjustment.py) through its own
    public API on the first `n_points` points of the workload: one constructor + optimize() call per
    entry of `calls` (iterations per call), exactly like the CUDA arm's chunks."""
    from oracle import build_ref

    RefBA = build_ref.load_reference_class()
    sc = sample_scene(name, n_points)
    x, vis = sc.dense_x()
    xt = np.ascontiguousarray(x.transpose(1, 0, 2)).transpose(1, 0, 2)  # as the scripts pass it
    done, t0 = 0, time.perf_counter()
    for m in calls:
        adj = RefBA(xt, sc.X0, sc.K0, sc.R0, sc.t0, f0=sc.f0, axis=sc.axis,
                    visibility_index=None if sc.dense else vis)
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            adj.optimize(SCALE, TOL_NEVER, max_iter=m)
        done += len(buf.getvalue().strip().splitlines())
    dt = time.perf_counter() - t0
    return {"value": sc.nobs * done / dt, "seconds": dt, "observations": sc.nobs, "iterations": done,
            "points": sc.n_points}


def reference_available(name: str = "c3") -> bool:
    """The unmodified reference can be timed: oracle/_ref is intact and the workload has a sample
    the reference can hold."""
    if REF_SAMPLE.get(name) is None:
        return False
    try:
        from oracle import build_ref

        return build_ref.verify()
    except Exception:
        return False


def cpu_baseline_leg(name: str, budget_iters: int = 8) -> dict:
    """cpu_baseline of the CUDA arm: the reference itself on a bounded sample (kind "reference");
    the port's figure on a larger sample rides along.  Falls back to the port alone when
    oracle/_ref was not built."""
    cores = use_all_host_threads()
    n_pts, iters = PORT_SAMPLE[name]
    port = oracle_port_run(name, n_pts, iters)
    port_desc = (f"{port['iterations']} LM iteration(s) of the CPU oracle port on the first {port['points']} points "
                 f"({port['observations']} observations) in {port['seconds']:.1f} s; {port['formulation']}")
    if reference_available(name):
        ref = reference_run(name, REF_SAMPLE[name], [budget_iters])
        return {"value": ref["value"], "unit": UNIT, "cores": cores, "kind": "reference",
                "sample": f"{ref['iterations']} LM iterations of the unmodified reference class (oracle/_ref) on the "
                          f"first {ref['points']} points x all cameras ({ref['observations']} observations) in "
                          f"{ref['seconds']:.1f} s; NumPy/BLAS with up to {blas_threads()} threads of {cores} cores "
                          "(the reference is effectively single-threaded outside BLAS)",
                "port": {"value": port["value"], "sample": port_desc}}
    return {"value": port["value"], "unit": UNIT, "cores": cores, "kind": "port", "sample": port_desc}


def run_reference(args, rank: int):
    """The reference arm: the reference's own CPU implementation of the path on the box's host
    cores -- the unmodified class from oracle/_ref when it was built, else the oracle port."""
    if rank != 0:
        return
    cores = use_all_host_threads()
    name = args.workload
    cfg = workload_config(name)
    K, W = args.steps, max(args.warmup, 0)
    calls = [min(CHUNK, K - k0) for k0 in range(0, K, CHUNK)]
    if reference_available(name):
        if W > 0:
            reference_run(name, REF_SAMPLE[name], [W])
        res = reference_run(name, REF_SAMPLE[name], calls)
        kind = "reference"
        sample = (f"{res['iterations']} LM iterations ({len(calls)} constructor + optimize() call(s)) of the unmodified "
                  f"reference class (oracle/_ref) on the first {res['points']} points x {cfg['n_cams']} cameras "
                  f"({res['observations']} observations) of {name}: the reference materialises an (N, n, n) float64 "
                  f"temporary (lib/bundle_adjustment.py:135), {8 * (9 * cfg['n_cams'] - 7) ** 2 / 1e6:.1f} MB per point; "
                  f"NumPy/BLAS, up to {blas_threads()} threads of {cores} cores")
    else:
        n_pts, _ = PORT_SAMPLE[name]
        if W > 0:
            oracle_port_run(name, n_pts, 1)
        res = oracle_port_run(name, n_pts, K if REF_SAMPLE.get(name) is not None else min(K, 3))
        kind = "port"
        sample = (f"{res['iterations']} LM iterations of the CPU oracle port on the first {res['points']} points "
                  f"({res['observations']} observations) of {name}; {res['formulation']}; {cores} cores"
                  + ("" if REF_SAMPLE.get(name) is not None else
                     "; the unmodified reference cannot hold a 1000-camera sample in which every camera is seen "
                     "(647 MB per point, singular system otherwise)"))
    out = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["seconds"] / max(res["iterations"], 1) * 1e3,
        "higher_is_better": True, "scaling": "weak" if args.weak else "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": describe(name, cfg, args.gpus, not args.weak),
        "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------------
class Ctx:
    """Process-wide handles of the CUDA arm."""

    def __init__(self, args, rank, world, local_rank):
        import torch

        import ba_b200

        self.args, self.rank, self.world, self.local_rank = args, rank, world, local_rank
        self.torch, self.ba = torch, ba_b200
        self.dist, self.group = None, None
        torch.cuda.set_device(local_rank)
        if world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
            self.dist, self.group = dist, dist.group.WORLD
        self.engine_mod = ba_b200.submodule("engine")
        self.sharded = ba_b200.submodule("sharded")
        self.gauge = ba_b200.submodule("gauge")

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v: float) -> float:
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())


def make_rank_scene(ctx: Ctx, name: str, strong: bool):
    cfg = workload_config(name)
    if ctx.world > 1 and strong:
        N = cfg["n_points"]
        lo, hi = N * ctx.rank // ctx.world, N * (ctx.rank + 1) // ctx.world
        sc = ctx.ba.scenes.make_scene(**{**cfg, "chunk_seeded": True}, point_range=(lo, hi))
    elif ctx.world > 1:
        sc = ctx.ba.scenes.make_scene(**cfg, point_stream=ctx.rank)
    else:
        sc = ctx.ba.scenes.make_scene(**cfg)
    return cfg, sc


def gather_scene_on_rank0(ctx: Ctx, sc):
    """The whole (strong-scaled) scene as CUDA tensors on rank 0: every rank contributes its shard
    over NCCL (padded all-gathers; the other ranks drop the result at once)."""
    torch, dist = ctx.torch, ctx.dist
    dev = f"cuda:{ctx.local_rank}"
    W = ctx.world
    counts = torch.tensor([sc.n_points, sc.nobs], dtype=torch.int64, device=dev)
    allc = torch.empty(2 * W, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(allc, counts)
    allc = allc.cpu().numpy().reshape(W, 2)
    max_pts, max_obs = int(allc[:, 0].max()), int(allc[:, 1].max())

    def gather(arr: np.ndarray, n_max: int, width: int, dtype):
        mine = torch.zeros((n_max, width) if width > 1 else (n_max,), dtype=dtype, device=dev)
        src = torch.from_numpy(np.ascontiguousarray(arr)).to(dev)
        mine[: src.shape[0]] = src
        out = torch.empty((W,) + tuple(mine.shape), dtype=dtype, device=dev)
        dist.all_gather_into_tensor(out, mine)
        return out if ctx.rank == 0 else None

    g_xy = gather(sc.obs_xy, max_obs, 2, torch.float64)
    g_cnt = gather(np.diff(sc.obs_ptr), max_pts, 1, torch.int64)
    g_X0 = gather(sc.X0, max_pts, 3, torch.float64)
    g_cam = None if sc.dense else gather(sc.obs_cam, max_obs, 1, torch.int32)
    if ctx.rank != 0:
        return None
    xy = torch.cat([g_xy[r, : allc[r, 1]] for r in range(W)]).contiguous()
    cnt = torch.cat([g_cnt[r, : allc[r, 0]] for r in range(W)])
    ptr = torch.zeros(cnt.shape[0] + 1, dtype=torch.int64, device=dev)
    ptr[1:] = torch.cumsum(cnt, 0)
    X0 = torch.cat([g_X0[r, : allc[r, 0]] for r in range(W)]).cpu().numpy()
    cam = None if g_cam is None else torch.cat([g_cam[r, : allc[r, 1]] for r in range(W)]).contiguous()
    return {"ptr": ptr, "cam": cam, "xy": xy, "X0": X0, "n_points": int(cnt.shape[0]), "n_obs": int(xy.shape[0])}


def single_gpu_trajectory(ctx: Ctx, sc, whole, iters: int, tol: float = TOL_NEVER):
    """Costs of the first `iters` LM iterations of the whole scene on rank 0's GPU alone."""
    eng = ctx.engine_mod.Engine(whole["n_points"], sc.n_cams, whole["n_obs"], sc.f0, sc.axis, sc.dense,
                                ctx.local_rank)
    eng.set_observations(whole["ptr"], whole["cam"], whole["xy"])
    Xn, Rn, tn = ctx.gauge.normalize(whole["X0"], sc.R0, sc.t0, sc.axis)
    eng.set_state(Xn, Rn, tn, np.ascontiguousarray(sc.K0[:, 0, 0]), np.ascontiguousarray(sc.K0[:, :2, 2]))
    recs, st = eng.lm_run(SCALE, tol, iters)
    E = [recs[0].E_prev] + [r.E for r in recs]
    eng.close()
    return np.array(E), int(st.solves)


def gather_rows_on_rank0(ctx: Ctx, arr: np.ndarray):
    """Every rank's rows of a float64 array, concatenated in rank order on rank 0 (None elsewhere)."""
    torch, dist, dev = ctx.torch, ctx.dist, f"cuda:{ctx.local_rank}"
    counts = torch.empty(ctx.world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(counts, torch.tensor([arr.shape[0]], dtype=torch.int64, device=dev))
    counts = counts.cpu().numpy()
    mine = torch.zeros((int(counts.max()),) + arr.shape[1:], dtype=torch.float64, device=dev)
    mine[: arr.shape[0]] = torch.from_numpy(np.ascontiguousarray(arr)).to(dev)
    out = torch.empty((ctx.world,) + tuple(mine.shape), dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(out, mine)
    if ctx.rank != 0:
        return None
    return np.concatenate([out[r, : counts[r]].cpu().numpy() for r in range(ctx.world)])


def dump_outputs(ctx: Ctx, adj, out_dir: str) -> None:
    """What the timed path computed in its last step, as optimize() hands it to its caller: X, K, R, t
    in the caller's frame, and E, the cost before and after every iteration of the last LM run, as
    out_dir/<name>.npy in float64.  At N > 1 the point shards are gathered on rank 0.  If the files
    would exceed DUMP_MAX_BYTES, X is a fixed seeded sample of rows, whose indices go to X_rows.npy."""
    eng = adj.engine
    X, R, t, f, u = eng.get_state(0)
    X, R, t = ctx.gauge.denormalize(adj._R0, adj._t0, adj._c0c1_len, X, R, t)
    recs = eng.lm_records()
    out = {"K": ctx.gauge.make_K(f, u, adj._f0), "R": R, "t": t,
           "E": np.array([recs[0].E_prev] + [r.E for r in recs])}
    if ctx.world > 1:
        X = gather_rows_on_rank0(ctx, X)
    if ctx.rank != 0:
        return
    budget = DUMP_MAX_BYTES - sum(a.nbytes for a in out.values())
    if X.nbytes > budget:
        rows = np.random.default_rng(DUMP_SEED).choice(X.shape[0], budget // (4 * 8), replace=False)
        rows.sort()
        X, out["X_rows"] = X[rows], rows.astype(np.float64)
    out["X"] = X
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def measure(ctx: Ctx, name: str, strong: bool, K: int, W: int, *, full_run_tol=None,
            with_e2e: bool = True, with_parity: bool = True, dump_dir: str | None = None) -> dict | None:
    """One workload on this invocation's ranks; rank 0 returns the result dict.  `full_run_tol`:
    instead of K steps in chunks, ONE optimize(2.0, tol, max_iter=K) call (config 5's convergence
    run).  `dump_dir`: write the outputs of the timed steps there (see dump_outputs)."""
    torch, args, rank, world, local_rank = ctx.torch, ctx.args, ctx.rank, ctx.world, ctx.local_rank
    dist, group, ba_b200 = ctx.dist, ctx.group, ctx.ba
    t_gen = time.perf_counter()
    cfg, sc = make_rank_scene(ctx, name, strong)
    t_gen = time.perf_counter() - t_gen
    convergence = full_run_tol is not None

    def pinned(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()

    h_ptr, h_xy = pinned(sc.obs_ptr), pinned(sc.obs_xy)
    h_cam = None if sc.dense else pinned(sc.obs_cam)
    h_X0, h_K0, h_R0, h_t0 = pinned(sc.X0), pinned(sc.K0), pinned(sc.R0), pinned(sc.t0)

    def make_adjuster(gauge_on_device=False):
        return ba_b200.BundleAdjuster.from_observations(
            h_ptr, h_cam, h_xy, h_X0, h_K0, h_R0, h_t0, f0=sc.f0, axis=sc.axis, dense=sc.dense,
            device=local_rank, process_group=group, exchange=args.exchange,
            gauge_on_device=gauge_on_device)

    def lm(adj, tol, m):
        eng = adj.engine
        if world > 1 and not adj._peer_exchange:
            st = ctx.sharded.lm_loop(eng, dist, group, SCALE, tol, m)
            return eng.lm_records(), st
        return eng.lm_run(SCALE, tol, m)

    def run_iters(adj, n):
        """Exactly n accepted LM iterations, as LM runs of at most CHUNK iterations, each started
        from the adjuster's initial state (kept on the device).  A run from the perturbed start
        needs ~14 iterations to reach the noise floor; there the accept test E_ > E is decided
        by the last bits of the cost sum, so the number of retries would depend on the summation
        order (hence on the GPU count) instead of on the work.  Chunks stay clear of the floor."""
        eng = adj.engine
        if getattr(adj, "_dev_init", None) is None:
            adj._dev_init = [torch.from_numpy(np.ascontiguousarray(a)).cuda(local_rank)
                             for a in (adj._X, adj._R, adj._t, adj._f, adj._u)]
        done, solves, st, first = 0, 0, None, None
        while done < n:
            m = min(CHUNK, n - done)
            eng.set_state(*adj._dev_init)
            recs, st = lm(adj, TOL_NEVER, m)
            assert st.count == m, f"ran {st.count} iterations instead of {m}"
            if first is None:
                first = [recs[0].E_prev] + [r.E for r in recs]
            done += m
            solves += st.solves
        st.solves, st.count = solves, done
        return st, np.array(first)

    # ---- device-resident arm ---------------------------------------------------------------
    adj = make_adjuster()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    traj = None
    if convergence:
        adj._dev_init = [torch.from_numpy(np.ascontiguousarray(a)).cuda(local_rank)
                         for a in (adj._X, adj._R, adj._t, adj._f, adj._u)]
        if W > 0:
            lm(adj, TOL_NEVER, min(W, 3))
            adj.engine.set_state(*adj._dev_init)
        ctx.barrier()
        launches0 = ctx.engine_mod.launch_count()
        t_wall0 = time.perf_counter()
        ev0.record()
        recs, st = lm(adj, full_run_tol, K)
        ev1.record()
        torch.cuda.synchronize()
        t_wall1 = time.perf_counter()
        traj = np.array([recs[0].E_prev] + [r.E for r in recs])
        steps_done = int(st.count)
    else:
        if W > 0:
            run_iters(adj, W)
        ctx.barrier()
        launches0 = ctx.engine_mod.launch_count()
        t_wall0 = time.perf_counter()
        ev0.record()
        st, traj = run_iters(adj, K)
        ev1.record()
        torch.cuda.synchronize()
        t_wall1 = time.perf_counter()
        steps_done = K
        assert st.count == K, f"ran {st.count} iterations instead of {K}"
    launches = ctx.engine_mod.launch_count() - launches0
    if dump_dir:
        dump_outputs(ctx, adj, dump_dir)
    ctx.barrier()
    ms = ctx.max_over_ranks(ev0.elapsed_time(ev1))
    nobs_total = int(ctx.sum_over_ranks(float(sc.nobs)))
    value = nobs_total * steps_done / (ms * 1e-3)
    final_rms = float(np.sqrt(st.E / nobs_total))
    exchange_desc = ("sums over NVLink peer memory by the library's kernels (CUDA-graph loop)"
                     if adj._peer_exchange else "two NCCL all-reduces per solve") if world > 1 else ""

    out = None
    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps_done, "warmup": W,
            "ms_per_step": ms / max(steps_done, 1), "higher_is_better": True,
            "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": describe(name, cfg, world, strong),
            "observations_total": nobs_total, "exchange": exchange_desc,
            "lm_iterations_per_s": steps_done / (ms * 1e-3), "inner_solves": int(st.solves),
            "final_rms": final_rms, "gpu_launches": int(launches), "scene_generation_s": t_gen,
        }
        if convergence:
            out["config"]["lm"] = (f"ONE optimize(2.0, {full_run_tol:g}, max_iter={K}) call from the perturbed start "
                                   "(BASELINE.json config 5's convergence run); one step = one accepted LM iteration")
            out["cost_first_last"] = [float(traj[0]), float(traj[-1])]

    # ---- roofline of the dominant kernel (rank 0, profiled re-run of the same K iterations) --
    if rank == 0 and world == 1 and not convergence:
        eng = adj.engine
        eng.profile_enable(True)
        eng.profile_reset()
        st_prof, _ = run_iters(adj, K)
        prof = eng.profile()
        eng.profile_enable(False)
        n_red = 9 * sc.n_cams - 7
        counts = np.diff(sc.obs_ptr)
        flops = float(np.sum(3.0 * (9.0 * counts) * (9.0 * counts + 1.0))) if not sc.dense else \
            3.0 * sc.n_points * n_red * (n_red + 1.0)
        peak = ctx.engine_mod.fp64_peak(local_rank, True)
        tot = sum(v["ms"] for k, v in prof.items() if k in ("k1", "k2", "k3", "k4", "cost", "other"))
        if sc.dense and prof["syrk"]["launches"] > 0:
            avg_ms = prof["syrk"]["ms"] / prof["syrk"]["launches"]
            kernel = "syrk_tma_kernel (K3, Schur SYRK on FP64 tensor cores, DMMA.8x8x4 fed by TMA)" \
                if ctx.engine_mod.syrk_feed() == "tma" else \
                "syrk_dmma_kernel (K3, Schur SYRK on FP64 tensor cores)"
            share = prof["syrk"]["ms"] / tot if tot > 0 else None
        else:
            avg_ms = prof["k3"]["ms"] / max(st_prof.solves, 1)
            kernel = "schur_pairs_kernel + schur_diag_kernel (K3, sparse Schur products, matrix-free pair kernel)"
            share = prof["k3"]["ms"] / tot if tot > 0 else None
        achieved = flops / (avg_ms * 1e-3) / 1e12
        out["roofline"] = {
            "kernel": kernel, "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
            "frac": achieved / peak, "traffic": None, "algorithmic_flops_per_launch": flops,
            "avg_launch_ms": avg_ms, "share_of_step": share,
            "operand_feed": ctx.engine_mod.syrk_feed() if sc.dense else None,
            "peak_source": "measured live: register-resident DMMA.8x8x4 loop (ba_fp64_peak); "
                           "MEASURED_PEAKS.json has no FP64 figure",
        }
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
                tr = json.load(f).get(name)
        except Exception:
            tr = None
        if tr:
            out["roofline"]["traffic"] = tr["dram_bytes_per_launch"]
            out["roofline"]["traffic_source"] = tr["source"]
        out["phase_ms_per_step"] = {k: v["ms"] / K for k, v in prof.items()}
        hbm = None
        try:
            hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs")
        except Exception:
            pass
        # memory-bound phases against the measured copy bandwidth (K1: 16 B read + 224 B written
        # per observation and linearisation)
        out["linearisation"] = ("matrix-free: K2a, camera blocks, K2b and the point update re-derive the Jacobian "
                                "rows; K1 stores nothing") if eng.matrix_free() else "K1 stores the Jacobian rows"
        if prof["k1"]["ms"] > 0 and not eng.matrix_free():
            gbs = sc.nobs * 240.0 * K / (prof["k1"]["ms"] * 1e-3) / 1e9
            out["k1_hbm"] = {"achieved_gbs": gbs, "peak_gbs": hbm or 6650.0,
                             "peak_source": "MEASURED_PEAKS.json" if hbm else "fallback",
                             "frac": gbs / (hbm or 6650.0), "bytes_per_obs": 240}

    if world > 1 and args.profile_ranks and adj._peer_exchange and not convergence:
        eng = adj.engine
        eng.profile_enable(True)
        eng.profile_reset()
        ctx.barrier()
        run_iters(adj, K)
        prof = eng.profile()
        eng.profile_enable(False)
        ctx.barrier()
        if rank == 0:
            out["phase_ms_per_step"] = {k: v["ms"] / K for k, v in prof.items()}

    # the device-resident engine is released first: the end-to-end arm re-creates one, as a
    # caller that adjusts scene after scene would
    adj.engine.close()
    del adj

    # ---- parity against one GPU on the same global scene (strong scaling only) ---------------
    if world > 1 and strong and with_parity and not args.no_parity:
        whole = gather_scene_on_rank0(ctx, sc)
        if rank == 0:
            # (a convergence run is compared over its first iterations only: close to the noise floor
            # the accept test is decided by the last bits of the cost sum, i.e. by the summation order)
            n_it = min(len(traj) - 1, CHUNK)
            E1, solves1 = single_gpu_trajectory(ctx, sc, whole, n_it, TOL_NEVER)
            m = min(len(E1), n_it + 1)
            rel = float(np.max(np.abs(traj[:m] - E1[:m]) / np.abs(E1[:m])))
            out["parity_vs_n1"] = {
                "max_rel_cost_diff": rel, "rtol": PARITY_RTOL, "iterations_compared": m - 1,
                "ok": bool(rel <= PARITY_RTOL and m == n_it + 1),
                "what": f"per-iteration cost of the run on {world} GPUs against a single-GPU run of the same global "
                        "scene made in this invocation on rank 0 (scene gathered over NCCL)"}
            del whole
        torch.cuda.empty_cache()
        ctx.barrier()

    # ---- end-to-end arm (host buffers in, host results out) ---------------------------------
    # Each repetition is the complete user call for K steps; the median of E2E_REPS wall times is
    # reported (all samples are listed), since a single cold call is dominated by allocator noise.
    if with_e2e:
        state_bytes = (3 * sc.n_points + 15 * sc.n_cams) * 8
        calls = [K] if convergence else [min(CHUNK, K - k0) for k0 in range(0, K, CHUNK)]
        tol = full_run_tol if convergence else TOL_NEVER
        obs_bytes = h_xy.nbytes + h_ptr.nbytes + (0 if h_cam is None else h_cam.nbytes)

        def timed_calls(make):
            samples, iters = [], 0
            for _ in range(E2E_REPS if not convergence else 1):
                ctx.barrier()
                t0 = time.perf_counter()
                iters = 0
                for m in calls:
                    adj2 = make()
                    with contextlib.redirect_stdout(io.StringIO()):
                        adj2.optimize(SCALE, tol, max_iter=m)
                    iters += len(adj2.records)
                    adj2.engine.close()
                torch.cuda.synchronize()
                samples.append(ctx.max_over_ranks(time.perf_counter() - t0))
            return samples, iters

        fo_samples, fo_iters = timed_calls(lambda: make_adjuster(gauge_on_device=True))
        fo_s = float(np.median(fo_samples))
        e2e = {"value": nobs_total * fo_iters / fo_s, "unit": UNIT,
               "h2d_bytes_per_step": len(calls) * (obs_bytes + state_bytes) / max(fo_iters, 1),
               "d2h_bytes_per_step": (len(calls) * state_bytes + fo_iters * 40) / max(fo_iters, 1),
               "ms_per_step": fo_s / max(fo_iters, 1) * 1e3,
               "samples_ms_per_step": [t / max(fo_iters, 1) * 1e3 for t in fo_samples],
               "what": f"{len(calls)} complete user call(s): BundleAdjuster.from_observations(pinned host arrays, "
                       "gauge_on_device=True).optimize(...): engine creation (device memory from the library's "
                       "retained pool), H2D of observations and state, gauge normalisation, LM iterations, "
                       f"de-normalisation, D2H of X/K/R/t; median of {len(fo_samples)} repetition(s)"}
        if sc.dense:
            # the reference's own signature: dense x (N, M, 2) handed over as np.stack(x_list).transpose(1, 0, 2)
            # (euclidiean_reconstruction.py:53-55), ordinary pageable arrays, host-side gauge passes
            x_cm = np.ascontiguousarray(sc.obs_xy.reshape(sc.n_points, sc.n_cams, 2).transpose(1, 0, 2))
            x_ref = x_cm.transpose(1, 0, 2)
            X0, K0, R0, t0 = (np.array(a) for a in (sc.X0, sc.K0, sc.R0, sc.t0))

            def make_ref_signature():
                return ba_b200.BundleAdjuster(x_ref, X0, K0, R0, t0, axis=sc.axis, device=local_rank,
                                              process_group=group, exchange=args.exchange)

            rs_samples, rs_iters = timed_calls(make_ref_signature)
            rs_s = float(np.median(rs_samples))
            e2e["from_observations"] = {k: e2e[k] for k in ("value", "ms_per_step", "samples_ms_per_step", "what",
                                                            "h2d_bytes_per_step", "d2h_bytes_per_step")}
            e2e.update({
                "value": nobs_total * rs_iters / rs_s, "ms_per_step": rs_s / max(rs_iters, 1) * 1e3,
                "samples_ms_per_step": [t / max(rs_iters, 1) * 1e3 for t in rs_samples],
                "h2d_bytes_per_step": len(calls) * (x_ref.nbytes + state_bytes) / max(rs_iters, 1),
                "what": f"{len(calls)} complete call(s) through the REFERENCE's constructor signature: "
                        "BundleAdjuster(x (N, M, 2) = np.stack(x_list).transpose(1, 0, 2), X, K, R, t, axis=...)"
                        ".optimize(...) with ordinary pageable NumPy arrays: engine creation, the camera-major block "
                        "uploaded as it lies in memory and re-ordered on the device, gauge normalisation and "
                        "de-normalisation in NumPy on the host, LM iterations, D2H of X/R/t/f/u; median of "
                        f"{len(rs_samples)} repetition(s)"})
        if rank == 0:
            out["e2e"] = e2e

    if rank == 0:
        out["_wall"] = (t_wall0, t_wall1)
    return out


def run_cuda(args, rank: int, world: int, local_rank: int):
    ctx = Ctx(args, rank, world, local_rank)
    strong = not args.weak
    K, W = args.steps, max(args.warmup, 0)
    name = args.workload

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    if name == "c5":
        out = measure(ctx, name, strong, K, W, full_run_tol=1e-8, dump_dir=args.dump_outputs)
    else:
        out = measure(ctx, name, strong, K, W, dump_dir=args.dump_outputs)
    if rank == 0:
        t_wall0, t_wall1 = out.pop("_wall")
        out["clocks"] = sampler.stop(t_wall0, t_wall1)

    # ---- extras ------------------------------------------------------------------------------
    if args.extras == "auto":
        extras = ["c2"] if world == 1 else (["c4", "c5"] if world == 8 else [])
    elif args.extras == "none":
        extras = []
    else:
        extras = [e for e in args.extras.split(",") if e]
    extras = [e for e in extras if e != name]
    extra = {}
    for e in extras:
        if e == "c5":
            res = measure(ctx, e, strong, 50, min(W, 3), full_run_tol=1e-8)
        else:
            res = measure(ctx, e, strong, min(K, 20) if e == "c2" else min(K, CHUNK), min(W, 3))
        if rank == 0:
            res.pop("_wall", None)
            key = e if world == 1 else f"{e}_n{world}"
            extra[key] = res

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            try:
                out["cpu_baseline"] = cpu_baseline_leg(name)
            except Exception as exc:  # the CPU leg must never cost the GPU line
                out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": None, "kind": "failed",
                                       "sample": f"{type(exc).__name__}: {exc}"}
        for key, res in extra.items():
            wl = key.split("_")[0]
            if wl in ("c4", "c5") and not args.no_cpu_baseline:
                # the sparsity-aware CPU denominator of the 1000-camera workloads (bounded sample)
                cores = use_all_host_threads()
                n_pts, iters = PORT_SAMPLE[wl]
                port = oracle_port_run(wl, n_pts, iters)
                res["cpu_baseline"] = {
                    "value": port["value"], "unit": UNIT, "cores": cores, "kind": "port",
                    "sample": f"{port['iterations']} LM iteration(s) ({port['solves']} solve(s)) on the first "
                              f"{port['points']} points x 1000 cameras ({port['observations']} observations) in "
                              f"{port['seconds']:.1f} s; {port['formulation']}; the unmodified reference needs 647 MB "
                              "per point here and is not a usable denominator",
                    "speedup_per_lm_iteration": res["value"] / port["value"]}
                if wl == "c5":
                    try:
                        with np.load(os.path.join(ROOT, "tests", "golden", "c5_shape.npz")) as z:
                            res["cpu_converged_rms"] = {
                                "value": float(z["rms"]),
                                "what": "converged RMS of the CPU oracle on a 5000-point scene of the same "
                                        "distribution (tests/golden/c5_shape.npz; the GPU reproduces that run to "
                                        "1e-9 in tests/test_gpu_parity.py) -- the 1M-point CPU run is out of reach"}
                    except Exception:
                        pass
        if extra:
            out["extra"] = extra
        print(json.dumps(out), flush=True)
        bad = [k for k, r in [("headline", out)] + list(extra.items())
               if r.get("parity_vs_n1") and not r["parity_vs_n1"]["ok"]]
        if bad:
            sys.stderr.write(f"parity_vs_n1 FAILED for {bad}\n")
    failed = False
    if rank == 0:
        failed = any(r.get("parity_vs_n1") and not r["parity_vs_n1"]["ok"] for r in [out] + list(extra.values()))
    if ctx.dist is not None:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()
    if failed:
        sys.exit(3)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world == 1 and args.gpus > 1:
        # not under torchrun: re-launch one rank per GPU
        port = 29500 + os.getpid() % 2000
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_cuda(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
