"""Write the outputs of the projective-depth iteration (primary and dual method) and of both rank-4
factorisations on fixed inputs as .npy files, so that two builds can be compared byte for byte
(`cmp`).  Set BA_DEPTH_JACOBI=1 to compare the Jacobi fallback of the eigenspace step as well.

    python tools/depth_outputs.py --out DIR

Host arrays in and out (BA_MEM_HOST), plus one run of every entry point on device arrays
(BA_MEM_DEVICE, files ending in `_dev`).
"""
import argparse
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import ba_b200  # noqa: E402


def scene_x(M, N, seed):
    sc = ba_b200.scenes.make_scene(M, N, seed=seed, visibility=1.0)
    xd, _ = sc.dense_x()
    return np.concatenate((xd / sc.f0, np.ones((N, M, 1))), axis=2), sc.f0


def seeded_w(n_rows, n_cols, seed):
    rs = np.random.RandomState(seed)
    low_rank = rs.standard_normal((n_rows, 4)) @ rs.standard_normal((4, n_cols))
    return low_rank + 1e-3 * rs.standard_normal((n_rows, n_cols))


def depth_on_device(symbol, x, f0, tol, iters):
    import torch

    cabi = ba_b200.submodule("_cabi")
    N, M = x.shape[:2]
    xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).cuda()
    zd = torch.empty((N, M), dtype=torch.float64, device="cuda")
    errors = np.empty(max(iters, 1), dtype=np.float64)
    n_iter = C.c_int(0)
    torch.cuda.synchronize()
    cabi.check(getattr(cabi.load(), symbol)(0, N, M, xd.data_ptr(), float(f0), float(tol), iters, zd.data_ptr(),
                                            errors.ctypes.data, C.byref(n_iter), cabi.BA_MEM_DEVICE, None))
    torch.cuda.synchronize()
    return zd.cpu().numpy(), errors[: n_iter.value].copy()


def factorize(W, centre, device_arrays):
    """(M, S, sigma[, mean]) straight from the C ABI."""
    cabi = ba_b200.submodule("_cabi")
    lib = cabi.load()
    n_rows, n_cols = W.shape
    Wt = np.ascontiguousarray(W.T)
    outs = [np.empty((n_rows, 4)), np.empty((4, n_cols)), np.empty(4)] + ([np.empty(n_rows)] if centre else [])
    if device_arrays:
        import torch

        dev = [torch.from_numpy(Wt).cuda()] + [torch.empty(o.shape, dtype=torch.float64, device="cuda") for o in outs]
        ptrs, mem = [t.data_ptr() for t in dev], cabi.BA_MEM_DEVICE
        torch.cuda.synchronize()
    else:
        ptrs, mem = [Wt.ctypes.data] + [o.ctypes.data for o in outs], cabi.BA_MEM_HOST
    if centre:
        w, m, s, sig, mean = ptrs
        cabi.check(lib.ba_factorize_centred_rank4(0, n_cols, n_rows, w, mean, m, s, sig, mem, None))
    else:
        w, m, s, sig = ptrs
        cabi.check(lib.ba_factorize_rank4(0, n_cols, n_rows, w, m, s, sig, mem, None))
    if device_arrays:
        torch.cuda.synchronize()
        outs = [t.cpu().numpy() for t in dev[1:]]
    return outs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    out = ap.parse_args().out
    os.makedirs(out, exist_ok=True)

    def save(name, *arrays, keys=("z", "errors")):
        for k, a in zip(keys, arrays):
            np.save(os.path.join(out, f"{name}_{k}.npy"), a)

    g = np.load(os.path.join(ROOT, "tests", "golden", "depth_primary.npz"))
    for c, iters in (("a", 200), ("b", 12)):
        x, f0, tol = g[c + "_x"], float(g[c + "_f0"]), float(g[c + "_tol"])
        save(f"primary_{c}", *ba_b200.projective_depth_primary(x, f0, tol, iters))
        if c == "b":
            save("primary_b_dev", *depth_on_device("ba_projective_depth_primary", x, f0, tol, iters))
    x, f0 = scene_x(50, 100_000, 1)
    save("primary_50x100k", *ba_b200.projective_depth_primary(x, f0, 0.0, 10))

    g = np.load(os.path.join(ROOT, "tests", "golden", "depth_dual.npz"))
    x, f0 = g["x"], float(g["f0"])
    save("dual_fixture", *ba_b200.projective_depth_dual(x, f0, float(g["tol"]), 50))
    save("dual_fixture15", *ba_b200.projective_depth_dual(x, f0, 1e-9, 15))
    save("dual_fixture15_dev", *depth_on_device("ba_projective_depth_dual", x, f0, 1e-9, 15))
    x, f0 = scene_x(40, 3000, 43)
    save("dual_40x3000", *ba_b200.projective_depth_dual(x, f0, 1e-12, 4))

    for name, W, centre in (("rank4_120x3000", seeded_w(120, 3000, 1), False),
                            ("rank4_192x20000", seeded_w(192, 20_000, 2), False),
                            ("centred_60x4000", seeded_w(60, 4000, 3) + 5.0, True)):
        keys = ("M", "S", "sigma", "mean")
        save(name, *factorize(W, centre, False), keys=keys)
        save(name + "_dev", *factorize(W, centre, True), keys=keys)
    print(f"wrote {len(os.listdir(out))} files to {out}")


if __name__ == "__main__":
    main()
