"""The emulated dense Schur product (Ozaki scheme II on the INT8 tensor cores) against an exact host
reconstruction, bit for bit.

Every step of the emulation before the final conversion is exact integer arithmetic, so P is fully
determined by Yt: the column scaling, the integer dot products modulo each p_i, Garner's digits, the
symmetric lift and the Horner evaluation with one rounding per fused multiply-add.  The host redoes
all of it from the Yt the engine used (read back from the device).  A k-block dropped or counted
twice by the int8 product changes P by far more than one unit in the last place, which a comparison
with the FP64 tensor-core product within a tolerance cannot see.

Shapes: n_pad < 256 (one ragged 256-tile); n_pad an exact multiple of 256; ragged last 256-tile rows
of 1, 9 and more than 128 rows of n = 9 M + 1; k_pad > 131 071 (several int32 accumulation runs per
tile); and a repeated build.  Needs a GPU."""
import numpy as np
import pytest
import torch

import ba_b200
from oracle import ba_oracle as O


def _engine_P_and_Yt(n_cams, n_points, monkeypatch, repeats=1):
    monkeypatch.setenv("BA_SYRK_EMU", "1")
    axis = "x-up_z-forward"
    sc = ba_b200.scenes.make_scene(n_cams, n_points, seed=n_cams + 7, visibility=1.0, axis=axis)
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr)),
                    sc.obs_cam.astype(np.int64), sc.obs_xy, sc.obs_ptr)
    X, R, t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, axis)
    eng = ba_b200.Engine(obs.n_points, obs.n_cams, obs.nobs, sc.f0, axis, True)
    try:
        assert eng.syrk_emulated()
        eng.set_observations(obs.ptr, None, obs.xy)
        eng.set_state(X, R, t, sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy())
        eng.linearize()
        Ps = []
        for _ in range(repeats):
            eng.build_reduced(1e-3)
            npad = eng.n_pad
            Ps.append(eng.buffer("REDUCE")[: npad * npad].reshape(npad, npad).copy())
        Yt = eng.buffer("YT").reshape(-1, npad)
        return Ps, Yt, eng.rhs_row
    finally:
        eng.close()


def _check_entries(n, rng, n_random=20_000):
    """Lower-triangle entries (rows, cols) to reconstruct: every row and column next to a 128-tile
    boundary and the last rows (the ragged tile row), plus a random sample.  A k-block dropped or
    doubled by a work item changes every entry of its tile."""
    edge = sorted({i for b in range(0, n + 128, 128) for i in (b - 1, b) if 0 <= i < n} | set(range(max(0, n - 16), n)))
    rows, cols = [], []
    for i in edge:
        rows += [i] * (i + 1)           # row i, columns 0..i
        cols += list(range(i + 1))
        rows += list(range(i, n))       # column i, rows i..n-1
        cols += [i] * (n - i)
    r = rng.integers(0, n, n_random)
    c = rng.integers(0, n, n_random)
    rows += np.maximum(r, c).tolist()
    cols += np.minimum(r, c).tolist()
    return np.unique(np.stack([rows, cols]), axis=1)


def _exact_P(Yt, moduli, bits, idx):
    """Entries idx = (rows, cols) of P = Yt^T Yt exactly as the emulation forms them."""
    k_pad, n_pad = Yt.shape
    # column exponents: the largest |entry| scaled below 2^bits (zero columns: exponent 0)
    cmax = np.abs(Yt).max(axis=0)
    e = np.where(cmax > 0, bits - 1 - (np.frexp(cmax)[1] - 1), 0).astype(np.int64)
    A = np.rint(np.ldexp(Yt, e[None, :]))  # integers of at most `bits` bits, exact in float64
    Ai = A.astype(np.int64)
    L = len(moduli)
    # residue sums: products of residues < 2^16 summed over k_pad < 2^37 rows are exact in float64 in
    # any order, so the device's FP64 product gives them exactly
    rows, cols = torch.from_numpy(idx[0]), torch.from_numpy(idx[1])
    x = np.empty((L, idx.shape[1]), dtype=np.int64)
    for i, p in enumerate(moduli):
        r = torch.from_numpy(np.mod(Ai, p).astype(np.float64)).cuda()
        x[i] = np.mod((r.T @ r).cpu()[rows, cols].numpy().astype(np.int64), p)
    # Garner's mixed-radix digits
    v = np.empty_like(x)
    for i, p in enumerate(moduli):
        t = x[i] % p
        for j in range(i):
            inv = pow(moduli[j], -1, p)
            t = ((t - v[j]) % p) * inv % p
        v[i] = t
    prod = 1
    for p in moduli:
        prod *= p
    half, hd = prod // 2, []
    for p in moduli:
        hd.append(half % p)
        half //= p
    # value >= prod / 2 is negative: compare digits from the most significant one
    cmp = np.zeros(idx.shape[1], dtype=np.int64)
    for i in range(L - 1, -1, -1):
        undecided = cmp == 0
        cmp[undecided & (v[i] > hd[i])] = 1
        cmp[undecided & (v[i] < hd[i])] = -1
    neg = cmp >= 0
    vl, nl = v, neg
    # Horner from the most significant digit; every step is __fma_rn(acc, p, d): the exact integer
    # acc * p + d (Python integers) rounded once to double
    acc = np.zeros(len(nl), dtype=object)
    vals = np.zeros(len(nl))
    for i in range(L - 1, -1, -1):
        d = np.where(nl, moduli[i] - 1 - vl[i] + (1 if i == 0 else 0), vl[i]).astype(object)
        vals = (acc * moduli[i] + d).astype(np.float64)
        acc = np.array([int(z) for z in vals.tolist()], dtype=object)
    vals = np.where(nl, -vals, vals)
    return np.ldexp(vals, -(e[idx[0]] + e[idx[1]]))


# (cameras, points): n = 9 M + 1 unknowns and rhs row, n_pad = n rounded up to 8
EXACT_SHAPES = [
    (17, 700),       # n_pad = 160 < 256: one ragged 256-tile
    (56, 600),       # n = 505, n_pad = 512: two full 256-tile rows
    (256, 120),      # n = 2305 = 9 x 256 + 1 (1 row past the last full tile row); n_pad 2312: ragged row of 8
    (200, 150),      # n = 1801 = 7 x 256 + 9; n_pad 1808: the headline shape's ragged row of 16
    (45, 44_000),    # n = 406 = 256 + 150 (> 128 rows); K = 132 000 > 131 071: two int32 runs per tile
    (1250, 300),     # n >> k, where the emulation is the default: n_pad = 11 256 = 43 x 256 + 248, k_pad = 928
                     # (2.2e6 entries checked: every 128-boundary row and column, ~15 s on the host)
]


@pytest.mark.gpu
@pytest.mark.parametrize("n_cams,n_points", EXACT_SHAPES)
def test_emulated_P_equals_exact_reconstruction(n_cams, n_points, monkeypatch):
    (P1, P2), Yt, rhs = _engine_P_and_Yt(n_cams, n_points, monkeypatch, repeats=2)
    moduli, bits = ba_b200.submodule("engine").syrk_emu_info(Yt.shape[0])
    n = rhs + 1
    idx = _check_entries(n, np.random.default_rng(n_cams))
    want = _exact_P(Yt, list(moduli), bits, idx)
    got = P1[idx[0], idx[1]]
    bad = np.flatnonzero(got.view(np.int64) != want.view(np.int64))
    assert bad.size == 0, (f"{bad.size} of {got.size} entries differ; first at ({idx[0][bad[0]]}, {idx[1][bad[0]]}): "
                           f"{got[bad[0]]!r} vs exact {want[bad[0]]!r}")
    assert np.array_equal(np.tril(P2[:n, :n]).view(np.int64), np.tril(P1[:n, :n]).view(np.int64)), \
        "a repeated build differs"
