"""The dense Schur product P = Yt^T Yt emulated on the INT8 tensor cores (Ozaki scheme II, K3).

Host part (CPU): the moduli and the bit budget the library reports, and a Python-integer restatement
of the arithmetic -- symmetric residues, Garner's mixed-radix conversion, the symmetric lift and the
Horner conversion to double -- against exact integer dot products.

GPU part: P from the emulated engine (BA_SYRK_EMU=1) against the same scene on the FP64 tensor cores
(BA_SYRK_EMU=0), exact zeros in the pinned gauge rows, and bitwise repeatability."""
import math

import numpy as np
import pytest

import ba_b200
from oracle import ba_oracle as O

C2_KPAD = 30016     # 50 cameras x 10 000 points: round_up(3 N, 32)
C3_KPAD = 300032    # 200 cameras x 100 000 points


def _kpad(n_points):
    return (3 * n_points + 31) // 32 * 32


def _info(k_pad):
    return ba_b200.submodule("engine").syrk_emu_info(k_pad)


@pytest.fixture(scope="module")
def built():
    import __graft_entry__

    __graft_entry__.build()


def test_moduli_are_pairwise_coprime_and_fit_int8(built):
    moduli, _ = _info(C3_KPAD)
    assert len(moduli) == 16
    assert all(2 <= p <= 256 for p in moduli)
    for i, p in enumerate(moduli):
        for q in moduli[i + 1:]:
            assert math.gcd(p, q) == 1, (p, q)


@pytest.mark.parametrize("k_pad", [C2_KPAD, C3_KPAD, _kpad(1500), _kpad(900), _kpad(333), _kpad(300),
                                   _kpad(50_000), 32])
def test_bit_budget_keeps_the_lift_exact(built, k_pad):
    moduli, b = _info(k_pad)
    half = math.prod(moduli) // 2
    assert 0 < b <= 53
    assert k_pad * 2 ** (2 * b) < half
    assert b == 53 or k_pad * 2 ** (2 * (b + 1)) >= half  # the largest such b
    if k_pad in (C2_KPAD, C3_KPAD):
        assert b == 53


def _sym_residue(a, p):
    """The kernel's residue: a - p rint(a / p), then 128 -> 128 - p (|r| <= 128 fits int8)."""
    q = (2 * a + p) // (2 * p)  # nearest integer (ties up; the kernel may differ by one there)
    r = a - p * q
    return r - p if r > 127 else r


def _lift(residue_sums, moduli):
    """Garner's mixed radix from the residue sums, symmetric lift, Horner in double from the top."""
    v = []
    for i, p in enumerate(moduli):
        t = residue_sums[i] % p
        for j in range(i):
            t = (t - v[j]) * pow(moduli[j], -1, p) % p
        v.append(t)
    prod = math.prod(moduli)
    value = sum(d * math.prod(moduli[:i]) for i, d in enumerate(v))
    neg = value >= prod // 2
    digits = [p - 1 - d for p, d in zip(moduli, v)] if neg else list(v)
    if neg:
        digits[0] += 1
    acc = 0.0
    for i in reversed(range(len(moduli))):
        acc = acc * float(moduli[i]) + float(digits[i])  # Python floats: one rounding per operation
    exact = value - prod if neg else value
    return (-acc if neg else acc), exact


@pytest.mark.parametrize("case", ["random", "edges", "negative", "zero"])
def test_residues_garner_and_lift_reproduce_exact_dot_products(built, case):
    k = 3000
    moduli, b = _info(_kpad(k // 3))
    rng = np.random.default_rng(7)
    top = 2 ** b
    if case == "random":
        a = [int(x) for x in rng.integers(-top, top, size=k, dtype=np.int64)]
        c = [int(x) for x in rng.integers(-top, top, size=k, dtype=np.int64)]
    elif case == "edges":  # every term at the largest magnitude: the sum reaches k 2^(2b)
        a = [top] * k
        c = [top] * k
    elif case == "negative":
        a = [-top] * k
        c = [top - int(x) for x in rng.integers(0, 1000, size=k)]
    else:
        a = [0] * k
        c = [top] * k
    exact = sum(x * y for x, y in zip(a, c))
    sums = []
    for p in moduli:
        ra = [_sym_residue(x, p) for x in a]
        rc = [_sym_residue(y, p) for y in c]
        assert all(-128 <= r <= 127 for r in ra + rc)
        # the int8 products accumulate exactly in int32 for <= 131 071 rows; each item's sum is
        # reduced mod p and added as an unsigned word
        s = sum(x * y for x, y in zip(ra, rc))
        assert abs(s) <= 128 * 128 * k
        sums.append(s % p)
    got, lifted = _lift(sums, moduli)
    assert lifted == exact
    if exact == 0:
        assert got == 0.0
    else:
        assert abs(got - exact) <= 16 * 2.0 ** -53 * abs(exact)


def test_lift_at_the_edges_of_the_symmetric_range(built):
    moduli, _ = _info(C3_KPAD)
    half = math.prod(moduli) // 2
    for x in (half - 1, -half, -1, 1, 2 ** 53, -(2 ** 53) - 1):
        got, lifted = _lift([x % p for p in moduli], moduli)
        assert lifted == x
        assert abs(got - x) <= 16 * 2.0 ** -53 * abs(x)


# ---- GPU ------------------------------------------------------------------------------------------

DENSE_SHAPES = [
    (30, 1500, "x-up_z-forward"),
    (120, 900, "x-right_z-forward"),
    (17, 333, "x-up_z-forward"),
    (260, 300, "x-right_z-forward"),
    (40, 50_000, "x-up_z-forward"),   # K = 150 000 > 131 071: two k pieces per tile
    (200, 300, "x-up_z-forward"),     # n_pad = 14 x 128 + 16: the DMMA reference runs tall 128-tiles
    (400, 700, "x-up_z-forward"),     # n_pad = 3608, k_pad = 2112: 128-tile DMMA reference
    (1250, 300, "x-up_z-forward"),    # n >> k (n_pad = 11 256, k_pad = 928): 43 full 256-tile rows and a
                                      # ragged row of 248, as the emulation is selected by default there
]


def _reduced_P(ba, sc, axis, emu, monkeypatch, c=1e-3, repeats=1):
    monkeypatch.setenv("BA_SYRK_EMU", "1" if emu else "0")
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr)),
                    sc.obs_cam.astype(np.int64), sc.obs_xy, sc.obs_ptr)
    X, R, t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, axis)
    f, u = sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy()
    eng = ba.Engine(obs.n_points, obs.n_cams, obs.nobs, sc.f0, axis, True)
    try:
        assert eng.syrk_emulated() == emu
        eng.set_observations(obs.ptr, None, obs.xy)
        eng.set_state(X, R, t, f, u)
        eng.linearize()
        out = []
        for _ in range(repeats):
            eng.build_reduced(c)
            npad = eng.n_pad
            out.append(eng.buffer("REDUCE")[: npad * npad].reshape(npad, npad).copy())
        return out, eng.rhs_row
    finally:
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_cams,n_points,axis", DENSE_SHAPES)
def test_emulated_schur_product_matches_dmma(n_cams, n_points, axis, monkeypatch):
    sc = ba_b200.scenes.make_scene(n_cams, n_points, seed=n_cams, visibility=1.0, axis=axis)
    assert sc.dense
    (P_ref,), rhs = _reduced_P(ba_b200, sc, axis, False, monkeypatch)
    (P1, P2), _ = _reduced_P(ba_b200, sc, axis, True, monkeypatch, repeats=2)
    n = rhs + 1  # unknowns and the rhs row
    low_ref, low1, low2 = (np.tril(P[:n, :n]) for P in (P_ref, P1, P2))
    scale = np.abs(low_ref).max()
    err = np.abs(low1 - low_ref).max()
    assert err <= 1e-13 * scale, f"max |P_emu - P_dmma| / max |P| = {err / scale:.3e}"
    removed, _ = O.gauge_indices(n_cams, axis)
    assert np.all(low1[removed, :] == 0) and np.all(low1[:, removed] == 0)
    assert np.array_equal(low1, low2), "two emulated builds of P differ"
