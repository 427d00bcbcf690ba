"""Kernel split of the dense Schur product emulated on the INT8 tensor cores (K3, Ozaki scheme II).

    python tools/syrk_emu_split.py [--cams 200] [--points 100000] [--reps 5] [--out DIR]

Builds the reduced system of one dense scene `reps` times on an engine created with BA_SYRK_EMU=1,
under torch.profiler (CUDA activities), and prints one JSON line: mean time per build of every K3
kernel and of K2b (k2b_point_solve_kernel, which gathers the column maxima the conversion needs; run
on a build before that change for K2b without them), the residue conversion's bandwidth (bytes it must
move: Yt read once, the residue planes written once), the int8 rate of both instances of syrk_i8_pair_kernel (whole tile rows, ragged last
tile row) and the operand bytes their TMA copies deliver to
shared memory per build.  The rate counts the MMA work the kernel issues: 2 x 256 x N x k per 256-tile
and modulus, N = 256 (diagonal tiles included: their upper halves are computed too), or the rows of a
ragged last tile row rounded up to 16.  The bytes are counted from the plan (a 128-row box of 128 k per
operand and CTA, one operand on a full diagonal tile), not profiled.  Needs a GPU."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _smi(field):
    import subprocess
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={field}", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out)
    except (OSError, ValueError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cams", type=int, default=200)
    ap.add_argument("--points", type=int, default=100_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for the Chrome trace")
    args = ap.parse_args()
    os.environ["BA_SYRK_EMU"] = "1"
    import torch
    from torch.profiler import ProfilerActivity, profile

    import ba_b200
    from oracle import ba_oracle as O

    sc = ba_b200.scenes.make_scene(args.cams, args.points, seed=1, visibility=1.0)
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr)),
                    sc.obs_cam.astype(np.int64), sc.obs_xy, sc.obs_ptr)
    X, R, t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, sc.axis)
    eng = ba_b200.Engine(obs.n_points, obs.n_cams, obs.nobs, sc.f0, sc.axis, True)
    assert eng.syrk_emulated()
    eng.set_observations(obs.ptr, None, obs.xy)
    eng.set_state(X, R, t, sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy())
    eng.linearize()
    eng.build_reduced(1e-3)  # warm-up
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.reps):
            eng.build_reduced(1e-3)
        torch.cuda.synchronize()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        prof.export_chrome_trace(os.path.join(args.out, "syrk_emu_split.pt.trace.json"))
    ms = {}
    for ev in prof.key_averages():
        name = ev.key
        if "syrk_i8_pair_kernel" in name:  # two instances: whole tile rows, and the ragged last tile row
            k = "syrk_i8_pair_kernel<ragged>" if "<true>" in name else "syrk_i8_pair_kernel<full>"
            ms[k] = ms.get(k, 0.0) + ev.device_time_total / 1e3 / args.reps
        for k in ("emu_residue_kernel", "emu_reconstruct_kernel", "k2b_point_solve_kernel"):
            if k in name:
                ms[k] = ms.get(k, 0.0) + ev.device_time_total / 1e3 / args.reps
        if "emset" in name:
            ms["memset"] = ms.get("memset", 0.0) + ev.device_time_total / 1e3 / args.reps
    n_pad, k_pad = eng.n_pad, (3 * args.points + 31) // 32 * 32
    moduli, bits = ba_b200.submodule("engine").syrk_emu_info(k_pad)
    nt2 = (n_pad + 255) // 256
    left = n_pad - (nt2 - 1) * 256
    thin_n = (left + 15) // 16 * 16
    full_rows = nt2 if left == 256 else nt2 - 1  # 256-tile rows without a ragged edge
    kb = (k_pad + 127) // 128
    scale = 16384.0 * kb * len(moduli)  # one 16 KB box (128 rows x 128 k) per k-block and modulus
    ops = {"full": 2.0 * 256 * 256 * full_rows * (full_rows + 1) // 2 * kb * 128 * len(moduli),
           "ragged": 0.0 if left == 256 else 2.0 * 256 * nt2 * thin_n * kb * 128 * len(moduli)}
    # operand boxes per k-block: off-diagonal 4, full diagonal 2, ragged row 4 (A tile + two B boxes)
    box_GB = {"full": (4 * (full_rows * (full_rows - 1) // 2) + 2 * full_rows) * scale / 1e9,
              "ragged": (0 if left == 256 else 4 * nt2) * scale / 1e9}
    # of which L2 -> SM: rows inside the tensor only (the ragged row's B boxes are mostly zero fill)
    l2_GB = dict(box_GB)
    if left != 256:
        l2_GB["ragged"] = nt2 * (2 * 16384.0 + 2 * 128.0 * min(left, 128)) * kb * len(moduli) / 1e9
    ki = {"full": "syrk_i8_pair_kernel<full>", "ragged": "syrk_i8_pair_kernel<ragged>"}
    conv_bytes = 8.0 * k_pad * n_pad + len(moduli) * float(n_pad) * k_pad
    conv_ms = ms.get("emu_residue_kernel", 0)
    k2b_ms = ms.pop("k2b_point_solve_kernel", None)
    res = {
        "scene": f"{args.cams} x {args.points}", "n_pad": n_pad, "k_pad": k_pad, "bits": bits, "moduli": len(moduli),
        "ms_per_build": ms,
        "syrk_total_ms": sum(ms.values()),
        "k2b_ms": k2b_ms,
        "conversion_bytes": conv_bytes,
        "conversion_GBps": conv_bytes / (conv_ms * 1e-3) / 1e9 if conv_ms else None,
        "i8_TOPS": {c: ops[c] / (ms[ki[c]] * 1e-3) / 1e12 for c in ops if ms.get(ki[c])},
        "i8_ops": ops,
        "tma_box_GB_per_build": box_GB,
        "l2_to_sm_GB_per_build": l2_GB,
        "gpu": torch.cuda.get_device_name(0),
        "power_limit_W": _smi("power.limit"), "sm_clock_MHz": _smi("clocks.sm"),
    }
    eng.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
