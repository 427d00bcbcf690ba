"""The reduced-system Cholesky (K4) on systems the test writes: backward error in every size regime,
and every way a pivot can fail.  The GPU tests need a B200 (`pytest -m gpu`); the bar and its
sensitivity are checked on the host.

The camera count M alone picks the regime (n = 9 M unknowns, n_rows = n + 1 with the rhs row):

    factorisation                                       back substitution         cameras
    one persistent cooperative launch (chol_fused)      one CTA                   M <= 113
    fused                                               8-CTA cluster             114 <= M <= 227
    two-level: chol_panel + rank-256 update, 64-tiles   whole grid                228 <= M <= 312
    two-level, first wide update on 128-tiles           grid                      M >= 313
      (n_rows - 256 >= kCholSplitMinRows)
    two-level                                           grid, more 64-blocks      M >= 1053
                                                        than the 148 SMs

Systems are written through the reduce buffer [P n_pad x n_pad | U M x 81 | d_F M x 9] between
lm_phase_reduce and lm_phase_solve, where a sharded run sums it over the ranks.  assemble_kernel
forms, on the lower triangle, S = U (1 + c) on the diagonal of the camera blocks minus P, the gauge
rows pinned to a unit diagonal, and b = P[rhs_row] - d_F.  A system A, b is written as P = -A,
U = 0, d_F = 0 with zero gauge rows and columns, so that the device assembles A exactly."""
import contextlib
import io
import re

import numpy as np
import pytest
import scipy.linalg as sl

from oracle import ba_oracle as O

U_RD = 2.0 ** -53                               # unit roundoff of float64
U_LD = float(np.finfo(np.longdouble).eps) / 2   # of the residual's accumulation
NB = 64                                         # kCholNB: panel and back-substitution block width
C_DAMP = 1e-4
SCALE = 2.0
BA_OK, BA_ERR_SINGULAR, BA_ERR_STALL = 0, 3, 6

gpu = pytest.mark.gpu


# ---- the bar ------------------------------------------------------------------------------------
# Work in the scaled system At = D^-1 A D^-1 (unit diagonal), xt = D x, rt = D^-1 r; then
# eta = max_i |rt_i| / ||xt||_1, the same number for A and for any D A D with D diagonal.  Rows of
# the scaled factor Lt have 2-norm <= 1 (to first order), so (|Lt| |Lt|^T)_ij <= 1 and for any
# vector v, || |Lt|^T |v| ||_2 <= ||v||_1.  With gamma_k = k u the device's rounding is, to first
# order (Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed., Thm 8.5, 10.3, Lemma 3.5):
#   1. factorisation  Lt Lt^T = At + dA, |dA| <= gamma_{n+1} |Lt||Lt^T|:     |dA xt|_i <= 1 n u ||xt||_1
#   2. the rhs row, swept along as row n (forward substitution): b = Lt y + db,
#      |db| <= gamma_{n+1} |Lt||y|, and ||y||_2 = ||Lt^T xt||_2 <= ||xt||_1:          1 n u ||xt||_1
#   3. the GEMV of the back substitution, rhs_B = y_B - L_CB^T x_C: its error s has
#      ||s||_2 <= gamma_n (||y||_2 + || |Lt^T||xt| ||_2), and |Lt s|_i <= ||s||_2:    2 n u ||xt||_1
#   4. x_B = W_B rhs_B with W_B = L_BB^-T formed by the panel kernel (the identity rows eliminated
#      like rows below the panel: a triangular solve per row, then one 64-long dot product per
#      entry): ||L_BB^T x_B - rhs_B||_2 <= 2 w u kappa_B ||rhs_B||_2, w <= min(n, 64) the block
#      width, kappa_B = cond_2(Lt_BB), and ||rhs_B||_2 = ||Lt_BB^T xt_B||_2 <= ||xt_B||_1:
#                                                                            2 n u kappa_B ||xt||_1
# Together eta <= (4 + 2 kappa_B) n u <= 6 n u max(1, kappa_B).  The reciprocal (rcp + two Newton
# steps) and rsqrt the kernels use for 1 / d_k and 1 / sqrt(d_k) are not correctly rounded: a few
# ulp per pivot, a relative error per entry of L that is O(u), not O(n u).  C = 8 leaves that and
# the second-order terms room.  The check's own rounding (residual accumulated in long double:
# gamma_{n+1} (|b| + |A||x|) <= 2 gamma_{n+1} in eta's units) is added to the bar.
C_ETA = 8.0


def eta_bar(n, kappa_b):
    return C_ETA * n * U_RD * max(1.0, kappa_b) + 2.0 * (n + 1) * U_LD


def backward_error(A, b, x):
    """eta = max_i |b - A x|_i / (d_i sum_j d_j |x_j|), d = sqrt(diag(A)); residual in long double."""
    d = np.sqrt(np.diag(A))
    xl = x.astype(np.longdouble)
    r = np.empty(b.size)
    for i in range(0, b.size, 1024):  # long double copies of a row block at a time
        r[i:i + 1024] = (b[i:i + 1024].astype(np.longdouble) - A[i:i + 1024].astype(np.longdouble) @ xl).astype(np.float64)
    return float(np.max(np.abs(r) / (d * np.sum(d * np.abs(x)))))


def scaled_factor(A):
    """Cholesky factor of D^-1 A D^-1 (host LAPACK)."""
    d = np.sqrt(np.diag(A))
    return np.linalg.cholesky(A / d[:, None] / d[None, :])


def block_kappa(L, n_full=None, kept=None):
    """Largest 2-norm condition number of the 64 x 64 diagonal blocks of L.  With `kept`, L is the
    factor on the kept unknowns of an n_full system whose gauge rows are identity rows; the blocks
    are those of the n_full system (a block's singular values are its kept part's and ones)."""
    if kept is None:
        n_full, kept = L.shape[0], np.arange(L.shape[0])
    worst = 1.0
    for b0 in range(0, n_full, NB):
        sel = np.flatnonzero((kept >= b0) & (kept < b0 + NB))
        if sel.size:
            worst = max(worst, float(np.linalg.cond(L[np.ix_(sel, sel)])))
    return worst


# ---- systems --------------------------------------------------------------------------------------
def spd_random(rng, n):
    """Q diag(lambda) Q^T, lambda log-uniform in [1, 1e3]; from n = 3000 on I + G G^T / 256 (O(n^2 256))."""
    if n > 3000:
        G = rng.standard_normal((n, 256))
        A = G @ G.T / 256.0
        A[np.diag_indices(n)] += 1.0
        return A
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    return _sym((Q * 10.0 ** rng.uniform(0.0, 3.0, n)) @ Q.T)


def spd_ill(rng, n):
    """Q diag(lambda) Q^T, lambda log-spaced from 1 to 1e13."""
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    return _sym((Q * np.logspace(0.0, 13.0, n)) @ Q.T)


def graded(rng, A):
    """D A D with D = diag(2^e), e uniform in [-30, 30]: exact in binary floating point."""
    D = np.ldexp(1.0, rng.integers(-30, 31, A.shape[0]))
    return A * D[:, None] * D[None, :], D


def _sym(A):
    return (A + A.T) / 2.0


def host_blocked_solve(A, b, drop=None):
    """The device's algorithm on the host: Cholesky, y = L^-1 b, then L^T x = y by 64-blocks from the
    last, rhs_B = y_B - sum_C L_CB^T x_C, x_B = W_B rhs_B with the explicit W_B = L_BB^-T.  `drop` =
    (C, B) leaves block L_CB out of the back substitution."""
    L = np.linalg.cholesky(A)
    y = sl.solve_triangular(L, b, lower=True)
    n = b.size
    x = np.zeros(n)
    nblk = (n + NB - 1) // NB
    for B in range(nblk - 1, -1, -1):
        b0, b1 = B * NB, min(n, B * NB + NB)
        rhs = y[b0:b1].copy()
        for Cb in range(B + 1, nblk):
            if drop != (Cb, B):
                c0, c1 = Cb * NB, min(n, Cb * NB + NB)
                rhs -= L[c0:c1, b0:b1].T @ x[c0:c1]
        W = sl.solve_triangular(L[b0:b1, b0:b1], np.eye(b1 - b0), lower=True).T
        x[b0:b1] = W @ rhs
    return x


# ---- regimes -----------------------------------------------------------------------------------------
SMS = 148                # B200
TWO_LEVEL_ROWS = 2048    # kCholTwoLevelRows
SPLIT_MIN_ROWS = 2560    # kCholSplitMinRows
OB = 256                 # kCholOB


def regime(M):
    """The K4 kernels a system of M cameras runs, from launch_cholesky_solve's size rules."""
    n = 9 * M
    n_rows = n + 1
    kernels = set()
    if n_rows < TWO_LEVEL_ROWS:
        kernels.add("chol_fused_kernel")
    else:
        kernels |= {"chol_panel_kernel", "chol_update_kernel"}
        for K0 in range(0, n, OB):
            if K0 + OB < n_rows:
                kernels.add("wide128" if n_rows - (K0 + OB) >= SPLIT_MIN_ROWS else "wide64")
    kernels.add("chol_backsolve_grid_kernel" if n >= 2048 else
                "chol_backsolve_cluster_kernel" if n >= 1024 else "chol_backsolve_kernel")
    return kernels


_K4_NAME = re.compile(r"\b(chol_\w+_kernel)\b")
_WIDE = re.compile(r"\bsyrk_(tma|dmma)_kernel\s*<\s*(true|1)\s*>")


def kernels_seen(names):
    seen = set()
    for name in names:
        m = _K4_NAME.search(name)
        if m:
            seen.add(m.group(1))
        m = _WIDE.search(name)
        if m:
            seen.add("wide128" if m.group(1) == "tma" else "wide64")
    return seen


ACCURACY_M = [2, 7, 8, 64, 113, 114, 227, 228, 320, 448, 1253]


# ---- host checks: the table, the bar and what it catches -------------------------------------------------
def test_accuracy_cases_cover_every_regime():
    """The camera counts of the accuracy cases reach every kernel of K4, both wide-update tile sizes,
    and a grid back substitution with more 64-blocks than SMs."""
    assert regime(113) == {"chol_fused_kernel", "chol_backsolve_kernel"}
    assert regime(114) == {"chol_fused_kernel", "chol_backsolve_cluster_kernel"}
    assert regime(227) == {"chol_fused_kernel", "chol_backsolve_cluster_kernel"}
    assert regime(228) == {"chol_panel_kernel", "chol_update_kernel", "wide64", "chol_backsolve_grid_kernel"}
    assert "wide128" not in regime(312) and "wide128" in regime(313)
    assert set().union(*map(regime, ACCURACY_M)) == {
        "chol_fused_kernel", "chol_panel_kernel", "chol_update_kernel", "wide64", "wide128",
        "chol_backsolve_kernel", "chol_backsolve_cluster_kernel", "chol_backsolve_grid_kernel"}
    assert max((9 * M + NB - 1) // NB for M in ACCURACY_M) > SMS
    assert min((9 * M + NB - 1) // NB for M in ACCURACY_M if M >= 1053) > SMS


@pytest.mark.parametrize("family", ["random", "graded", "ill"])
@pytest.mark.parametrize("n", [63, 576, 2052])
def test_bar_holds_for_the_algorithm_on_the_host(family, n):
    """The host's run of the same algorithm (explicit inverses of the diagonal blocks) stays under
    the bar on every family."""
    rng = np.random.default_rng(n)
    A = spd_ill(rng, n) if family == "ill" else spd_random(rng, n)
    b = rng.standard_normal(n)
    if family == "graded":
        A, D = graded(rng, A)
        b = b * D
    x = host_blocked_solve(A, b)
    kappa = block_kappa(scaled_factor(A))
    eta = backward_error(A, b, x)
    assert eta <= eta_bar(n, kappa), (family, n, eta, eta_bar(n, kappa), kappa)


def _coupled_system(rng, n, eps):
    """Well-conditioned 64-blocks (eigenvalues in [1, 10]) coupled by entries of size eps."""
    A = eps * rng.standard_normal((n, n))
    A = _sym(A)
    for b0 in range(0, n, NB):
        w = min(NB, n - b0)
        Q, _ = np.linalg.qr(rng.standard_normal((w, w)))
        A[b0:b0 + w, b0:b0 + w] = _sym((Q * rng.uniform(1.0, 10.0, w)) @ Q.T)
    return A


def test_eta_catches_a_dropped_block_of_the_factor():
    """Leaving one off-diagonal 64 x 64 block of L out of the back substitution moves the step by
    less than the 1e-8 max|dxi| that the scene comparisons allow, and fails the eta bar."""
    rng = np.random.default_rng(1)
    n = 3 * NB
    A = _coupled_system(rng, n, 2e-9)
    b = rng.standard_normal(n)
    x = host_blocked_solve(A, b)
    bar = eta_bar(n, block_kappa(scaled_factor(A)))
    assert backward_error(A, b, x) <= bar
    x_bad = host_blocked_solve(A, b, drop=(2, 0))
    assert np.max(np.abs(x_bad - x)) <= 1e-8 * np.max(np.abs(x))
    eta = backward_error(A, b, x_bad)
    assert eta > bar, (eta, bar)


def test_eta_catches_noise_in_one_block_of_the_step():
    """Noise of 1e-11 max|x| on the 64 entries of the block that carries the step passes the 1e-8
    step comparison and fails the eta bar.  The step's entries span three decades, as a BA step's
    do (focal lengths in pixels, rotations in radians)."""
    rng = np.random.default_rng(2)
    n = 2 * NB
    A = _coupled_system(rng, n, 1e-2)
    x_true = np.concatenate((1e-3 * rng.standard_normal(NB), rng.choice([-1.0, 1.0], NB) * 10.0 ** rng.uniform(-3, 0, NB)))
    b = A @ x_true
    x = host_blocked_solve(A, b)
    bar = eta_bar(n, block_kappa(scaled_factor(A)))
    assert backward_error(A, b, x) <= bar
    x_bad = x.copy()
    x_bad[NB:] += 1e-11 * np.max(np.abs(x)) * rng.choice([-1.0, 1.0], NB)
    assert np.max(np.abs(x_bad - x)) <= 1e-8 * np.max(np.abs(x))
    eta = backward_error(A, b, x_bad)
    assert eta > bar, (eta, bar)


# ---- the device harness ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ba():
    import ba_b200

    return ba_b200


class System:
    """A dense engine of M cameras (40 points: the points only have to exist) and torch views of its
    reduce buffer.  begin() puts it back into its initial state."""

    def __init__(self, ba, M):
        sc = ba.scenes.make_scene(M, 40, seed=M, visibility=1.0)
        X, R, t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, sc.axis)
        self.state = (X, R, t, sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy())
        self.M, self.n, self.axis = M, 9 * M, sc.axis
        self.removed, self.kept = O.gauge_indices(M, sc.axis)
        self.eng = ba.Engine(sc.n_points, M, sc.nobs, sc.f0, sc.axis, True)
        self.eng.set_observations(sc.obs_ptr, None, sc.obs_xy)
        npad = self.eng.n_pad
        red = self.eng.reduce_tensor()
        self.P = red[: npad * npad].view(npad, npad)
        self.U = red[npad * npad: npad * npad + 81 * M].view(M, 9, 9)
        self.dF = red[npad * npad + 81 * M: npad * npad + 90 * M]

    def begin(self, max_retries=200):
        self.eng.set_state(*self.state)
        self.eng.lm_begin(SCALE, 1e-8, 10, max_retries)

    def reduce(self):
        import torch

        self.eng.lm_phase_reduce()
        torch.cuda.synchronize()

    def solve(self):
        import torch

        torch.cuda.synchronize()
        self.eng.lm_phase_solve()

    def own_system(self, c):
        """(A, b) on the kept unknowns, formed from the buffer as assemble_kernel forms them."""
        n, M = self.n, self.M
        P = self.P[: n + 1, : n + 1].cpu().numpy()
        U = self.U.cpu().numpy()
        dF = self.dF.cpu().numpy()
        A = -np.tril(P[:n, :n])
        del P
        for i in range(M):
            blk = np.tril(U[i])
            blk[np.diag_indices(9)] *= 1.0 + c
            A[9 * i: 9 * i + 9, 9 * i: 9 * i + 9] += blk
        A += np.tril(A, -1).T
        k = self.kept
        b = self.P[n, :n].cpu().numpy()[k] - dF[k]
        return A[np.ix_(k, k)], b

    def write_system(self, A, b):
        """P = -A and rhs row b on the kept unknowns, zero gauge rows and columns, U = 0, d_F = 0."""
        import torch

        n, k = self.n, self.kept
        full = np.zeros((n, n))
        full[np.ix_(k, k)] = -A
        rhs = np.zeros(n)
        rhs[k] = b
        torch.cuda.synchronize()
        self.P[:n, :n].copy_(torch.from_numpy(full))
        self.P[n, :n].copy_(torch.from_numpy(rhs))
        self.U.zero_()
        self.dF.zero_()
        torch.cuda.synchronize()


_SYSTEMS = {}


@pytest.fixture(scope="module")
def system(ba):
    def get(M):
        if M not in _SYSTEMS:
            _SYSTEMS[M] = System(ba, M)
        return _SYSTEMS[M]
    yield get
    for s in _SYSTEMS.values():
        s.eng.close()
    _SYSTEMS.clear()


# ---- accuracy: scaled backward error in every regime ----------------------------------------------------
FAMILIES = ["own", "random", "graded", "ill"]


def _accuracy_cases():
    for M in ACCURACY_M:
        for fam in FAMILIES:
            if fam == "ill" and M == 1253:
                continue  # Q diag(lambda) Q^T is O(n^3) on the host at n = 11 270; the others cover M
            yield M, fam


@gpu
@pytest.mark.parametrize("M,family", list(_accuracy_cases()))
def test_backward_error(system, M, family):
    """eta of the device's step against C n u max(1, kappa_B), whatever cond(A); on the ill-conditioned
    family also the forward error against cond(D^-1 A D^-1) times that bar.  The graded system is
    the random one scaled by powers of two, which every operation of K4 carries exactly: its step is
    the random system's step times D^-1, bit for bit."""
    s = system(M)
    s.begin()
    s.reduce()
    rng = np.random.default_rng(10 * M + FAMILIES.index("random" if family == "graded" else family))
    nk = s.kept.size
    if family == "own":
        A, b = s.own_system(C_DAMP)
    else:
        A = spd_ill(rng, nk) if family == "ill" else spd_random(rng, nk)
        b = rng.standard_normal(nk)
        if family == "graded":
            s.write_system(A, b)
            s.solve()
            x_ungraded = s.eng.buffer("DXI")[s.kept]
            A, D = graded(rng, A)
            b = b * D
    s.write_system(A, b)
    s.solve()
    st = s.eng.lm_state()
    dxi = s.eng.buffer("DXI")
    assert st.chol_fail == 0 and st.status == BA_OK
    assert np.all(dxi[s.removed] == 0.0)
    x = dxi[s.kept]
    Ls = scaled_factor(A)
    kappa = block_kappa(Ls, s.n, s.kept)
    eta = backward_error(A, b, x)
    bar = eta_bar(s.n, kappa)
    print(f"M={M} {family}: eta {eta:.3e} bar {bar:.3e} kappa_B {kappa:.3e}")
    assert eta <= bar, f"M = {M} ({sorted(regime(M))}), {family}: eta {eta:.3e} > bar {bar:.3e} (kappa_B {kappa:.3e})"
    if family == "graded":
        moved = np.flatnonzero(x * D != x_ungraded)
        assert moved.size == 0, f"M = {M}: {moved.size} entries of D x differ from the ungraded step, first {moved[:5]}"
    if family == "ill":
        d = np.sqrt(np.diag(A))
        cf = (Ls, True)
        bt = b / d
        xr = sl.cho_solve(cf, bt)
        At = A / d[:, None] / d[None, :]
        r = (bt.astype(np.longdouble) - At.astype(np.longdouble) @ xr.astype(np.longdouble)).astype(np.float64)
        xr = xr + sl.cho_solve(cf, r)  # scaled reference, one refinement step
        ev = np.linalg.eigvalsh(At)
        cond = ev[-1] / ev[0]
        fwd = np.linalg.norm(d * x - xr) / np.linalg.norm(xr)
        print(f"M={M} ill: forward {fwd:.3e} bar {cond * bar:.3e} cond {cond:.3e}")
        assert fwd <= cond * bar, f"M = {M}: forward error {fwd:.3e} > {cond * bar:.3e} (cond {cond:.3e})"


@gpu
def test_accuracy_cases_reach_every_kernel(system):
    """The solves of the accuracy cases' camera counts, under the profiler: every kernel of K4 runs,
    both wide-update tile sizes among them.  One profiler session for all of them: in a run of the
    whole suite, one session per small solve came back without some of its kernels.  The first
    camera count is solved once more at the end, so that no record the check needs is the last."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    for M in ACCURACY_M:
        system(M).begin()
        system(M).reduce()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for M in ACCURACY_M + ACCURACY_M[:1]:
            system(M).solve()
        torch.cuda.synchronize()
    names = {ev.key for ev in prof.key_averages()}
    want = set().union(*map(regime, ACCURACY_M))
    assert kernels_seen(names) == want, f"ran {sorted(kernels_seen(names))}, want {sorted(want)}"


# ---- non-positive pivots and the LM decision ------------------------------------------------------
FAIL_M = [60, 227, 228, 320]


def _columns(M):
    """First kept column, the panel and outer-block edges, one inside the last panel, and (M = 320)
    one after the first 128-tile wide update."""
    n = 9 * M
    last = (n - 1) // NB * NB
    cols = [0, 63, 64, 255, 256, (last + n) // 2]
    return cols + [300] if M == 320 else cols


def _inject(s, kind, r, c):
    """Make pivot r negative (S_rr = -A_rr), exactly zero (row and column r of P and of the camera's U
    block) or NaN (one NaN at P[r][r - 1]; P[0][0] for r = 0)."""
    import torch

    i, a = divmod(r, 9)
    torch.cuda.synchronize()
    if kind == "negative":
        s.P[r, r] += 2.0 * (s.U[i, a, a] * (1.0 + c) - s.P[r, r])
    elif kind == "zero":
        s.P[r, :] = 0.0
        s.P[:, r] = 0.0
        s.U[i, a, :] = 0.0
        s.U[i, :, a] = 0.0
    else:
        s.P[r, max(r - 1, 0)] = float("nan")
    torch.cuda.synchronize()


def _state_equal(s):
    return all(np.array_equal(a, b) for a, b in zip(s.eng.get_state(0), s.state))


def _assert_rejected(s, st, solves=1, c=C_DAMP * SCALE):
    assert (st.chol_fail, st.status, st.accepted, st.count, st.solves, st.need_linearize, st.done) == \
        (1, BA_OK, 0, 0, solves, 0, 0), _fields(st)
    assert st.c == c
    assert _state_equal(s)


def _assert_singular(s, st):
    assert (st.status, st.done, st.accepted, st.count, st.solves) == (BA_ERR_SINGULAR, 1, 0, 0, 1), _fields(st)
    assert _state_equal(s)


def _fields(st):
    return {k: getattr(st, k) for k, _ in st._fields_}


_AFTER_REJECT = {}


def _after_reject_reference(ba, s):
    """DXI and trial cost of a fresh engine's build_reduced / solve_trial at the doubled damping."""
    if s.M not in _AFTER_REJECT:
        fresh = System(ba, s.M)
        fresh.eng.set_state(*fresh.state)
        fresh.eng.cost(0)  # the camera table of the state, as lm_begin forms it
        fresh.eng.linearize()
        fresh.eng.build_reduced(C_DAMP * SCALE)
        fresh.eng.solve_trial(C_DAMP * SCALE)
        _AFTER_REJECT[s.M] = (fresh.eng.buffer("DXI"), fresh.eng.cost_values()[1])
        fresh.eng.close()
    return _AFTER_REJECT[s.M]


@gpu
@pytest.mark.parametrize("kind", ["negative", "zero", "nan"])
@pytest.mark.parametrize("M,r", [(M, r) for M in FAIL_M for r in _columns(M)])
def test_bad_pivot(ba, system, M, r, kind):
    """A negative pivot rejects the step and doubles the damping; a zero or NaN pivot stops the run
    as singular.  After a reject the next solve, on the Lt / Winv / ywork the poisoned one filled with
    NaN, gives bit for bit what a fresh engine gives at the doubled damping (the LM phases and the
    single-phase entry points run the same kernels on the same inputs)."""
    s = system(M)
    s.begin()
    s.reduce()
    _inject(s, kind, r, C_DAMP)
    s.solve()
    s.eng.lm_phase_decide()
    st = s.eng.lm_state()
    if kind != "negative":
        _assert_singular(s, st)
        return
    _assert_rejected(s, st)
    s.reduce()
    s.solve()
    dxi, e_trial = s.eng.buffer("DXI"), s.eng.cost_values()[1]
    s.eng.lm_phase_decide()
    st = s.eng.lm_state()
    assert st.chol_fail == 0 and st.status == BA_OK and st.solves == 2
    ref_dxi, ref_e = _after_reject_reference(ba, s)
    assert np.all(np.isfinite(dxi))
    assert dxi.tobytes() == ref_dxi.tobytes()
    assert e_trial == ref_e


COMBOS = {
    # (kind, column) pairs: the first failing panel reports, inside a panel the lowest column
    "negative, zero in a later outer block": ([("negative", 64), ("zero", 300)], "reject"),
    "zero, negative in a later outer block": ([("zero", 64), ("negative", 300)], "singular"),
    "negative below zero, one panel": ([("negative", 70), ("zero", 100)], "reject"),
    "zero below negative, one panel": ([("zero", 70), ("negative", 100)], "singular"),
}


@gpu
@pytest.mark.parametrize("combo", list(COMBOS))
@pytest.mark.parametrize("M", FAIL_M)
def test_two_bad_pivots(system, M, combo):
    s = system(M)
    injections, outcome = COMBOS[combo]
    s.begin()
    s.reduce()
    for kind, r in injections:
        _inject(s, kind, r, C_DAMP)
    s.solve()
    s.eng.lm_phase_decide()
    st = s.eng.lm_state()
    if outcome == "reject":
        _assert_rejected(s, st)
    else:
        _assert_singular(s, st)


@gpu
@pytest.mark.parametrize("M", FAIL_M)
def test_pinned_rows_ignore_their_diagonal(system, M):
    """assemble_kernel writes 1 on a gauge row's diagonal whatever P holds there."""
    import torch

    s = system(M)
    s.begin()
    s.reduce()
    s.solve()
    ref = s.eng.buffer("DXI")
    assert np.all(np.isfinite(ref))
    s.begin()
    s.reduce()
    torch.cuda.synchronize()
    for r in s.removed:
        s.P[r, r] = -1e300
    s.solve()
    assert s.eng.buffer("DXI").tobytes() == ref.tobytes()
    assert s.eng.lm_state().chol_fail == 0


@gpu
@pytest.mark.parametrize("M", FAIL_M)
def test_retry_cap_on_negative_pivots(system, M):
    """A negative pivot on every solve: BA_ERR_STALL after max_retries solves, the damping doubled on
    each, the state untouched."""
    s = system(M)
    s.begin(max_retries=3)
    c = C_DAMP
    for k in range(3):
        s.reduce()
        _inject(s, "negative", 64, c)
        s.solve()
        s.eng.lm_phase_decide()
        st = s.eng.lm_state()
        c *= SCALE
        assert st.c == c and st.chol_fail == 1 and st.solves == k + 1 and st.accepted == 0, _fields(st)
    assert (st.status, st.done, st.count) == (BA_ERR_STALL, 1, 0), _fields(st)
    assert st.c == C_DAMP * 8
    assert _state_equal(s)


# ---- a camera nobody sees, in the two-level regime -------------------------------------------------------
@gpu
@pytest.mark.parametrize("M,blind", [(240, 7), (240, 28), (240, 239), (320, 7), (320, 28), (320, 319)])
def test_blind_camera_is_singular_in_the_two_level_regime(ba, M, blind):
    """The camera's rows are all zero; its first kept row is an exactly zero pivot in the panel kernel
    (camera 7: rows 63..71 straddle a panel edge, camera 28: rows 252..260 an outer-block edge).
    optimize raises the reference's LinAlgError on the first solve, and so does the covariance."""
    sc = ba.scenes.make_scene(M, 450, seed=M, visibility=0.3)
    pt = np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr))
    keep = sc.obs_cam != blind
    pt, cam, xy = pt[keep], sc.obs_cam[keep], sc.obs_xy.reshape(-1, 2)[keep]
    views = np.bincount(pt, minlength=sc.n_points)
    assert views.min() >= 2
    ptr = np.concatenate(([0], np.cumsum(views))).astype(np.int64)
    adj = ba.BundleAdjuster.from_observations(ptr, cam, xy, sc.X0, sc.K0, sc.R0, sc.t0, f0=sc.f0, axis=sc.axis)
    assert adj.engine.n_full + 1 >= TWO_LEVEL_ROWS
    with pytest.raises(np.linalg.LinAlgError, match="Singular matrix"):
        with contextlib.redirect_stdout(io.StringIO()):
            adj.optimize(SCALE, 1e-8, max_iter=5)
    st = adj.engine.lm_state()
    assert st.solves == 1 and st.count == 0
    with pytest.raises(np.linalg.LinAlgError):
        adj.engine.covariance()
    adj.engine.close()
