"""Kernel split of the dense Schur product emulated on the INT8 tensor cores (K3, Ozaki scheme II).

    python tools/syrk_emu_split.py [--cams 200] [--points 100000] [--reps 5] [--out DIR]

Builds the reduced system of one dense scene `reps` times on an engine created with BA_SYRK_EMU=1,
under torch.profiler (CUDA activities), and prints one JSON line: mean time per build of every K3
kernel, the conversion passes' bandwidth (bytes they must move: Yt read twice, the residue planes
written once) and the int8 rate of syrk_i8_kernel (2 x 128 x N x k ops per MMA tile, N = 128, or 16
on a ragged last tile row).  Needs a GPU."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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
        for k in ("emu_colmax_kernel", "emu_residue_kernel", "syrk_i8_kernel", "emu_reconstruct_kernel"):
            if k in name:
                ms[k] = ms.get(k, 0.0) + ev.device_time_total / 1e3 / args.reps
        if "emset" in name:
            ms["memset"] = ms.get("memset", 0.0) + ev.device_time_total / 1e3 / args.reps
    n_pad, k_pad = eng.n_pad, (3 * args.points + 31) // 32 * 32
    moduli, bits = ba_b200.submodule("engine").syrk_emu_info(k_pad)
    nt1 = (n_pad + 127) // 128
    left = n_pad - (nt1 - 1) * 128
    thin_n = 128 if left == 128 else (left + 15) // 16 * 16
    tiles_n = (nt1 - 1) * nt1 // 2 * 128 + nt1 * thin_n  # sum of N over the lower tiles
    kb = (k_pad + 127) // 128 * 128
    i8_ops = 2.0 * 128 * tiles_n * kb * len(moduli)
    conv_bytes = 2 * 8.0 * k_pad * n_pad + len(moduli) * float(n_pad) * k_pad
    conv_ms = ms.get("emu_colmax_kernel", 0) + ms.get("emu_residue_kernel", 0)
    res = {
        "scene": f"{args.cams} x {args.points}", "n_pad": n_pad, "k_pad": k_pad, "bits": bits, "moduli": len(moduli),
        "ms_per_build": ms,
        "syrk_total_ms": sum(ms.values()),
        "conversion_GBps": conv_bytes / (conv_ms * 1e-3) / 1e9 if conv_ms else None,
        "residue_pass_GBps": (8.0 * k_pad * n_pad + len(moduli) * float(n_pad) * k_pad)
        / (ms["emu_residue_kernel"] * 1e-3) / 1e9 if ms.get("emu_residue_kernel") else None,
        "i8_TOPS": i8_ops / (ms["syrk_i8_kernel"] * 1e-3) / 1e12 if ms.get("syrk_i8_kernel") else None,
        "i8_ops": i8_ops,
        "gpu": torch.cuda.get_device_name(0),
    }
    eng.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
