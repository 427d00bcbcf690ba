"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the reference's golden
vectors.  Everything here needs a B200: `pytest -m gpu`.

Bars (BASELINE.json north_star): per-iteration cost within 1e-9 relative, final points and
cameras within 1e-6; per-kernel quantities are compared much tighter (1e-11 .. 1e-12 relative
to their scale) because they are single float64 expressions."""
import contextlib
import io

import numpy as np
import pytest

from conftest import RUN_CASES, SMALL_CASES, case_inputs, load_golden
from oracle import ba_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ba():
    import ba_b200

    return ba_b200


def _engine_for(ba, obs: O.ObsList, X, R, t, f, u, f0, axis, dense):
    Engine = ba.Engine
    eng = Engine(obs.n_points, obs.n_cams, obs.nobs, f0, axis, dense)
    eng.set_observations(obs.ptr, None if dense else obs.cam.astype(np.int32), obs.xy)
    eng.set_state(X, R, t, f, u)
    return eng


def _close(a, b, rel, what):
    scale = max(np.abs(b).max(), 1e-300)
    err = np.abs(a - b).max() / scale
    assert err <= rel, f"{what}: max err / scale = {err:.3e} > {rel:.1e}"


def _check_linearisation(ba, obs, X, R, t, f, u, f0, axis, dense):
    """cost(0), K1 and K2 against the oracle; returns the linearised engine and the oracle's
    linearisation."""
    N, M = obs.n_points, obs.n_cams
    eng = _engine_for(ba, obs, X, R, t, f, u, f0, axis, dense)
    lin = O.linearize(obs, X, f, u, R, t, f0)

    # a20: cost
    assert eng.cost(0) == pytest.approx(O.cost(obs, X, f, u, R, t, f0), rel=1e-13)

    # K1: residuals + Jacobians
    eng.linearize()
    JP = eng.buffer("JP").reshape(-1, 8)
    JC = eng.buffer("JC").reshape(-1, 20)
    _close(JP[:, :2], lin.e, 1e-12, "residual (JP)")
    _close(JC[:, :2], lin.e, 1e-12, "residual (JC)")
    _close(JP[:, 2:].reshape(-1, 2, 3), lin.Jx, 1e-12, "de/dX")
    _close(JC[:, 2:].reshape(-1, 2, 9), lin.Jc, 1e-12, "de/dcam")

    # K2: point blocks, camera blocks (gauge rows zeroed)
    V = eng.buffer("V").reshape(N, 6)
    iu = ([0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2])
    _close(V, lin.V[:, iu[0], iu[1]], 1e-12, "V_j")
    _close(eng.buffer("GPT").reshape(N, 3), lin.g_pt, 1e-11, "d_P")
    removed, kept = O.gauge_indices(M, axis)
    # the diagonal blocks U_i, entries in kept rows and columns (block by block: the 9M x 9M block
    # diagonal is a gigabyte from 1250 cameras on)
    keep = np.zeros(9 * M, dtype=bool)
    keep[kept] = True
    keep = keep.reshape(M, 9)
    keep = keep[:, :, None] & keep[:, None, :]
    U = eng.buffer("U").reshape(M, 9, 9)
    _close(U[keep], lin.U[keep], 1e-12, "U_i")
    assert np.all(U[~keep] == 0)
    g = eng.buffer("GCAM")
    _close(g[kept], lin.g_cam.ravel()[kept], 1e-11, "d_F")
    assert np.all(g[removed] == 0)
    return eng, lin


def _check_one_linearisation(ba, obs, X, R, t, f, u, f0, axis, dense, c=1e-4):
    M = obs.n_cams
    eng, lin = _check_linearisation(ba, obs, X, R, t, f, u, f0, axis, dense)
    removed, kept = O.gauge_indices(M, axis)

    # K2b + K3: partial reduced system P = sum Y Y^T with the rhs row.  From n ~ 10^4 the oracle forms
    # the reduced system with its C restatement and solves it by Cholesky (the dense route and LU take
    # minutes there); either way it is formed once and the solve below reuses it.
    schur, solver = ("sparse", "cholesky") if 9 * M > 10_000 else ("dense", "lu")
    reduced = O.reduced_system_sparse(obs, lin, c) if schur == "sparse" else O.reduced_system(obs, lin, c)
    A_ref, b_ref, _ = reduced
    eng.build_reduced(c)
    red = eng.buffer("REDUCE")
    npad, nfull, rhs = eng.n_pad, eng.n_full, eng.rhs_row
    P = red[: npad * npad].reshape(npad, npad)
    b_gpu = P[rhs, :nfull] - red[npad * npad + 81 * M:]
    _close(b_gpu[kept], b_ref[kept], 1e-10, "reduced rhs b")
    # A = blockdiag(U_i with the diagonal scaled by 1 + c) - P, formed in place (n^2 doubles at a time)
    A_gpu = np.tril(P[:nfull, :nfull])
    A_gpu += np.tril(A_gpu, -1).T
    assert np.all(A_gpu[removed] == 0)
    np.negative(A_gpu, out=A_gpu)
    Ured = red[npad * npad: npad * npad + 81 * M].reshape(M, 9, 9)
    for i in range(M):
        blk = Ured[i].copy()
        blk[np.arange(9), np.arange(9)] *= 1 + c
        A_gpu[9 * i: 9 * i + 9, 9 * i: 9 * i + 9] += blk
    _close(A_gpu[np.ix_(kept, kept)], A_ref[np.ix_(kept, kept)], 1e-11, "reduced system A")
    del P, A_gpu

    # K4: solve, update, trial cost
    dxi_ref, dX_ref, _, _ = O.solve_damped(obs, lin, c, axis, solver=solver, reduced=reduced)
    eng.solve_trial(c)
    dxi = eng.buffer("DXI").reshape(M, 9)
    _close(dxi, dxi_ref, 1e-8, "camera step")
    assert np.all(dxi.ravel()[removed] == 0)
    tX, tR, tt, tf, tu = eng.get_state(1)
    rX, rf, ru, rR, rt = O.apply_update(X, f, u, R, t, dxi_ref, dX_ref)
    _close(tX, rX, 1e-9, "trial X")
    _close(tR, rR, 1e-9, "trial R")
    _close(tt, rt, 1e-9, "trial t")
    _close(tf, rf, 1e-9, "trial f")
    np.testing.assert_allclose(tu, ru, rtol=0, atol=1e-9)
    E_trial = float(eng.cost_values()[1])
    assert E_trial == pytest.approx(O.cost(obs, rX, rf, ru, rR, rt, f0), rel=1e-8)
    eng.close()
    return E_trial, red


@pytest.mark.parametrize("name", SMALL_CASES)
def test_kernels_match_oracle_on_golden_cases(ba, name):
    g = load_golden(name)
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    obs = O.ObsList.from_dense(x, vis)
    X, R, t = O.normalize_gauge(X0, R0, t0, axis)
    f, u = K0[:, 0, 0].copy(), K0[:, :2, 2].copy()
    E_trial, _ = _check_one_linearisation(ba, obs, X, R, t, f, u, f0, axis, dense=vis is None)
    # and against the reference's own first trial cost
    assert E_trial == pytest.approx(float(g["lin_E_trial"]), rel=1e-8)


def _check_random_scene(ba, n_cams, n_points, visibility, axis):
    sc = ba.scenes.make_scene(n_cams, n_points, seed=n_cams, visibility=visibility, axis=axis)
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr)),
                    sc.obs_cam.astype(np.int64), sc.obs_xy, sc.obs_ptr)
    X, R, t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, axis)
    f, u = sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy()
    return _check_one_linearisation(ba, obs, X, R, t, f, u, sc.f0, axis, dense=sc.dense)


# (cameras, points, visibility) past the camera-count thresholds that select kernel instances
# (test_camera_count_limits.py checks that these scenes reach every instance).  Seed = cameras;
# cond(S) at the initial state and c = 1e-4: 9.9e4, 3.9e5, 1.1e5, 1.1e5.  1253 cameras because seed
# 1250 leaves a camera barely constrained (cond(S) = 3.5e8).
CAMERA_COUNT_SCENES = [
    (361, 500, 1.0),    # the largest matrix-free dense engine: 48 KB camera table, 121 KB of shared
                        # memory in the point update
    (400, 700, 1.0),    # dense on stored rows (K1 writes them), camera table in shared memory,
                        # 128-tile DMMA SYRK, two-level Cholesky with 128-tile updates
    (1253, 300, 1.0),   # dense, camera table in global memory, emulated SYRK at n >> k (n_pad = 11 280,
                        # k_pad = 928), 177 64-blocks on at most 148 back-substitution CTAs
    (1253, 2000, 0.1),  # the same for the list engine and its pair lists
]


# Sparse scenes run twice: with the static pair lists (schur_pairs_reg_kernel) and with
# BA_PAIRS_NO_LIST (schur_pairs_kernel scans the bitmaps: the path of scenes whose lists do not fit).
@pytest.mark.parametrize("n_cams,n_points,visibility,axis,lists", [
    (30, 1500, 1.0, "x-up_z-forward", True),      # dense, 64-wide SYRK tiles, several k splits
    (120, 900, 1.0, "x-right_z-forward", True),   # dense, 128-wide SYRK tiles, multi-panel Cholesky
    (40, 2000, 0.3, "x-up_z-forward", True),      # sparse path
    (40, 2000, 0.3, "x-up_z-forward", False),
    (17, 333, 1.0, "x-up_z-forward", True),       # ragged sizes (nothing a multiple of anything)
    (70, 3000, 0.9, "x-up_z-forward", True),      # sparse path, nearly full bitmaps, 3 x 3 pair tiles
    (70, 3000, 0.9, "x-up_z-forward", False),     # bitmap scan: multi-pass hit queue
    (33, 200, 0.5, "x-right_z-forward", True),    # sparse path, one camera beyond a pair tile
    (33, 200, 0.5, "x-right_z-forward", False),   # bitmap scan: single bitmap batch
    (5, 9000, 0.7, "x-up_z-forward", True),       # sparse path, few cameras, long pair lists
    (5, 9000, 0.7, "x-up_z-forward", False),      # bitmap scan: several bitmap batches per pair
    (320, 450, 0.3, "x-up_z-forward", True),      # n = 2880: two-level Cholesky (rank-256 DMMA updates, 128- and 64-tiles), grid-wide back substitution
    (320, 450, 0.3, "x-up_z-forward", False),
    (260, 300, 1.0, "x-right_z-forward", True),   # n = 2340, dense: same with 64-tiles only, edge tiles cut by n_rows
    (1000, 1500, 0.1, "x-up_z-forward", True),    # C4's camera count: n = 8993, 35 outer blocks of the two-level Cholesky,
                                                  # 141-CTA back substitution, 31 x 31 pair tiles (oracle: ~25 s of LU)
    *[(m, n, v, "x-up_z-forward", True) for m, n, v in CAMERA_COUNT_SCENES],
])
def test_kernels_match_oracle_on_random_scenes(ba, monkeypatch, n_cams, n_points, visibility, axis, lists):
    if not lists:
        monkeypatch.setenv("BA_PAIRS_NO_LIST", "1")
    _check_random_scene(ba, n_cams, n_points, visibility, axis)


def test_bitmap_scan_pair_kernel_is_the_one_that_ran(ba, monkeypatch):
    """BA_PAIRS_NO_LIST really switches the pair kernel: the list kernel sums on per-lane FMA chains, the
    bitmap scan on DMMA fragments, so the two reduced systems differ in the last bits somewhere, and
    both match the oracle."""
    _, red_lists = _check_random_scene(ba, 70, 3000, 0.9, "x-up_z-forward")
    monkeypatch.setenv("BA_PAIRS_NO_LIST", "1")
    _, red_scan = _check_random_scene(ba, 70, 3000, 0.9, "x-up_z-forward")
    assert not np.array_equal(red_lists, red_scan)


@pytest.mark.parametrize("n_cams,n_points,axis", [
    (30, 1500, "x-up_z-forward"),
    (120, 900, "x-right_z-forward"),
    (17, 333, "x-up_z-forward"),
    (400, 700, "x-up_z-forward"),    # dense engine on stored rows, camera table in shared memory
    (1250, 300, "x-up_z-forward"),   # both engines read the camera table from global memory; seed 1253:
                                     # cond(S) = 1.1e5 at c = 1e-4
])
def test_matrix_free_linearisation_is_bitwise_the_stored_row_one(ba, n_cams, n_points, axis):
    """A dense engine of at most 361 cameras re-derives the Jacobian rows in K2a, the camera blocks,
    K2b and the point update (ba_matrix_free); a larger one stores them in K1 and reads them back, as
    an engine built from the same observations as a LIST always does.  The arithmetic is shared and
    pinned (obs_jacobian, scaled_point_rows, y_entry, pair_accumulate in ba_common.cuh) and the
    summation orders coincide for full visibility, so V, d_P, U, d_F, L^-1 and z must agree bit for
    bit -- as must the rows that the matrix-free engine writes on request (JP / JC buffer reads)."""
    sc = ba.scenes.make_scene(n_cams, n_points, seed=3 + n_cams, visibility=1.0, axis=axis)
    assert sc.dense
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr)),
                    sc.obs_cam.astype(np.int64), sc.obs_xy, sc.obs_ptr)
    X, R, t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, axis)
    f, u = sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy()
    dn = _engine_for(ba, obs, X, R, t, f, u, sc.f0, axis, dense=True)
    ls = _engine_for(ba, obs, X, R, t, f, u, sc.f0, axis, dense=False)
    assert dn.matrix_free() == (n_cams <= 361) and not ls.matrix_free()
    for eng in (dn, ls):
        eng.linearize()
        eng.build_reduced(1e-3)
    for name in ("V", "GPT", "U", "GCAM", "LINV", "Z", "JP", "JC"):
        a, b = dn.buffer(name), ls.buffer(name)
        assert np.array_equal(a, b), f"{name}: {np.abs(a - b).max():.3e}"
    # the reduced systems come from different Schur kernels (SYRK / pair products): equal to rounding;
    # the dense engine keeps P = Y Y^T with the rhs in row 9M, the list engine the same layout
    npad, n, rhs = dn.n_pad, dn.n_full, dn.rhs_row
    assert (npad, n, rhs) == (ls.n_pad, ls.n_full, ls.rhs_row)
    Pa = dn.buffer("REDUCE")[: npad * npad].reshape(npad, npad)
    Pb = ls.buffer("REDUCE")[: npad * npad].reshape(npad, npad)
    _close(np.tril(Pa[:n, :n]), np.tril(Pb[:n, :n]), 1e-12, "P (lower triangle)")
    _close(Pa[rhs, :n], Pb[rhs, :n], 1e-12, "rhs row")
    # one step: the same trial state (the matrix-free point update re-derives Y, the others read it)
    for eng in (dn, ls):
        eng.solve_trial(1e-3)
    for got, ref, what in zip(dn.get_state(1), ls.get_state(1), ("X", "R", "t", "f", "u")):
        _close(got, ref, 1e-11, f"trial {what}")
    dn.close()
    ls.close()


@pytest.mark.parametrize("name", RUN_CASES)
@pytest.mark.parametrize("debug", [False, True])
def test_full_run_matches_reference_golden(ba, name, debug):
    g = load_golden(name)
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    adj = ba.BundleAdjuster(x, X0, K0, R0, t0, f0=f0, visibility_index=vis, axis=axis)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        X, K, R, t = adj.optimize(2.0, 1e-8, max_iter=100, is_debug=debug)
    E = np.array([adj.records[0]["E_prev"]] + [r["E"] for r in adj.records])
    assert E.shape == g["E"].shape, "different number of accepted iterations"
    np.testing.assert_allclose(E, g["E"], rtol=1e-9, atol=0)
    np.testing.assert_allclose(X, g["X"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(K, g["K"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(R, g["R"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(t, g["t"], rtol=0, atol=1e-6)
    ref_lines = str(g["stdout"]).strip().splitlines()
    got_lines = buf.getvalue().strip().splitlines()
    assert len(got_lines) == len(ref_lines)
    for a, b in zip(got_lines, ref_lines):
        pa, pb = a.split(" = "), b.split(" = ")
        assert pa[0] == pb[0]
        assert float(pa[1]) == pytest.approx(float(pb[1]), rel=1e-6, abs=1e-12)
    if debug:
        log = adj.get_log()
        assert len(log) == len(g["E"])
        np.testing.assert_allclose(np.stack([d["points"] for d in log]), g["log_points"], rtol=0, atol=1e-6)
        np.testing.assert_allclose(np.stack([d["basis"] for d in log]), g["log_basis"], rtol=0, atol=1e-6)
        np.testing.assert_allclose(np.stack([d["pos"] for d in log]), g["log_pos"], rtol=0, atol=1e-6)
        np.testing.assert_allclose([d["reprojection_error"] for d in log], g["E"], rtol=1e-9)
    else:
        assert adj.get_log() == []


@pytest.mark.parametrize("visibility", [1.0, 0.4])
def test_graph_loop_equals_eager_loop(ba, visibility, monkeypatch):
    """ba_lm_run replays one captured CUDA graph per inner solve, one solve ahead of the host;
    BA_NO_GRAPH=1 keeps the launches eager.  Same kernels, same order: bit-identical records,
    also when the engine (and its graphs) is reused for a second run."""
    import os

    sc = ba.scenes.make_scene(12, 400, seed=5, visibility=visibility)
    runs = []
    for no_graph in (False, True, False):
        if no_graph:
            monkeypatch.setenv("BA_NO_GRAPH", "1")
        else:
            monkeypatch.delenv("BA_NO_GRAPH", raising=False)
        assert (os.environ.get("BA_NO_GRAPH") == "1") == no_graph
        adj = ba.BundleAdjuster.from_observations(sc.obs_ptr, sc.obs_cam, sc.obs_xy, sc.X0, sc.K0, sc.R0,
                                                  sc.t0, f0=sc.f0, axis=sc.axis, dense=sc.dense)
        eng = adj.engine
        for rep in range(2):
            eng.set_state(adj._X, adj._R, adj._t, adj._f, adj._u)
            recs, st = eng.lm_run(2.0, 1e-8, 30)
            runs.append(([(r.E_prev, r.E, r.c, r.solves) for r in recs], st.solves, eng.get_state(0)[0].copy()))
        eng.close()
    for other in runs[1:]:
        assert other[0] == runs[0][0]
        assert other[1] == runs[0][1]
        assert np.array_equal(other[2], runs[0][2])


@pytest.mark.parametrize("name", ["small_flip_xup", "small_sparse_xright", "c1_euclid"])
def test_gauge_on_device_matches_reference_golden(ba, name):
    """SURVEY.md 8f row 1: normalise / de-normalise (:208-258) as CUDA kernels, including the
    reference's negative-divisor quirk (small_flip_xup)."""
    g = load_golden(name)
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    adj = ba.BundleAdjuster(x, X0, K0, R0, t0, f0=f0, visibility_index=vis, axis=axis, gauge_on_device=True)
    # the normalised state the kernels produced against the host mirror of the reference's transform
    Xn, Rn, tn = ba.submodule("gauge").normalize(X0, R0, t0, axis)
    dX, dR, dt, _, _ = adj.engine.get_state(0)
    np.testing.assert_allclose(dX, Xn, rtol=0, atol=1e-13 * max(1.0, np.abs(Xn).max()))
    np.testing.assert_allclose(dR, Rn, rtol=0, atol=1e-14)
    np.testing.assert_allclose(dt, tn, rtol=0, atol=1e-13 * max(1.0, np.abs(tn).max()))
    with contextlib.redirect_stdout(io.StringIO()):
        X, K, R, t = adj.optimize(2.0, 1e-8, max_iter=100)
    E = np.array([adj.records[0]["E_prev"]] + [r["E"] for r in adj.records])
    assert E.shape == g["E"].shape
    np.testing.assert_allclose(E, g["E"], rtol=1e-9, atol=0)
    np.testing.assert_allclose(X, g["X"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(K, g["K"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(R, g["R"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(t, g["t"], rtol=0, atol=1e-6)


def test_inputs_are_not_written(ba):
    """The affine script passes a read-only broadcast K (reference affine_reconstruction.py:45)."""
    g = load_golden("small_dense_xup")
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    K_ro = np.broadcast_to(np.eye(3), K0.shape)
    copies = [a.copy() for a in (x, X0, R0, t0)]
    adj = ba.BundleAdjuster(x.transpose(1, 0, 2).copy().transpose(1, 0, 2), X0, K_ro, R0, t0, axis=axis)
    with contextlib.redirect_stdout(io.StringIO()):
        adj.optimize(2.0, 1e-8, max_iter=5)
    for a, b in zip((x, X0, R0, t0), copies):
        assert np.array_equal(a, b)


def test_error_behaviour(ba):
    g = load_golden("small_sparse_xup")
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    with pytest.raises(ValueError):
        ba.BundleAdjuster(x, X0, K0, R0, t0, axis="z-up")
    # a point without any view: the reference's inv() raises LinAlgError (:128)
    vis2 = vis.copy()
    vis2[3, :] = False
    adj = ba.BundleAdjuster(x, X0, K0, R0, t0, visibility_index=vis2, axis=axis)
    with pytest.raises(np.linalg.LinAlgError):
        with contextlib.redirect_stdout(io.StringIO()):
            adj.optimize(2.0, 1e-8, max_iter=5)


def test_observation_list_constructor_equals_dense_constructor(ba):
    g = load_golden("small_sparse_xright")
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    obs = O.ObsList.from_dense(x, vis)
    adj = ba.BundleAdjuster.from_observations(obs.ptr, obs.cam, obs.xy, X0, K0, R0, t0, axis=axis)
    with contextlib.redirect_stdout(io.StringIO()):
        X, K, R, t = adj.optimize(2.0, 1e-8, max_iter=100)
    np.testing.assert_allclose(X, g["X"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(K, g["K"], rtol=0, atol=1e-6)


def test_full_size_c2_properties(ba):
    """Config 2 (50 cameras x 10k points, dense) is beyond what the oracle checks in seconds
    per iteration end to end, so it is checked through size-independent properties: first
    iterations against the oracle, monotone cost, converged RMS at the injected noise level,
    and idempotence (re-optimising the optimum moves nothing)."""
    sc = ba.scenes.make_scene(**ba.scenes.CONFIGS["c2"])
    adj = ba.BundleAdjuster.from_observations(sc.obs_ptr, sc.obs_cam, sc.obs_xy, sc.X0, sc.K0, sc.R0,
                                              sc.t0, f0=sc.f0, axis=sc.axis, dense=True)
    with contextlib.redirect_stdout(io.StringIO()):
        X, K, R, t = adj.optimize(2.0, 1e-8, max_iter=100)
    E = np.array([adj.records[0]["E_prev"]] + [r["E"] for r in adj.records])
    assert np.all(np.diff(E) <= 0)
    rms = np.sqrt(E[-1] / sc.nobs)
    assert 0.8 * 0.005 * np.sqrt(2) < rms < 1.2 * 0.005 * np.sqrt(2)
    # two oracle iterations from the same start
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), sc.n_cams),
                    np.tile(np.arange(sc.n_cams), sc.n_points), sc.obs_xy, sc.obs_ptr)
    ora = O.OracleBundleAdjuster(None, sc.X0, sc.K0, sc.R0, sc.t0, f0=sc.f0, axis=sc.axis, obs=obs)
    ora.optimize(2.0, 1e-8, max_iter=2, verbose=False)
    Eo = np.array([r["E"] for r in ora.trace])
    np.testing.assert_allclose(E[:3], Eo, rtol=1e-9)
    # idempotence
    adj2 = ba.BundleAdjuster.from_observations(sc.obs_ptr, sc.obs_cam, sc.obs_xy, X, K, R, t, f0=sc.f0,
                                               axis=sc.axis, dense=True)
    with contextlib.redirect_stdout(io.StringIO()):
        X2, K2, R2, t2 = adj2.optimize(2.0, 1e-8, max_iter=100)
    assert len(adj2.records) <= 3
    assert adj2.records[-1]["E"] == pytest.approx(E[-1], rel=1e-7)
    # compare in the normalised gauge (the reference's sign quirk, :228-234, can reflect the
    # scene when the output is fed back in, so the caller's frame is not a fixed point)
    nX, nR, nt = O.normalize_gauge(X, R, t, sc.axis)
    nX2, nR2, nt2 = O.normalize_gauge(X2, R2, t2, sc.axis)
    np.testing.assert_allclose(np.abs(nX2), np.abs(nX), rtol=0, atol=1e-5)
    np.testing.assert_allclose(np.abs(nt2), np.abs(nt), rtol=0, atol=1e-5)


def test_full_size_c3_properties(ba):
    """Config 3 (200 cameras x 100k points, dense: 2e7 observations, n = 1793) at full size.  The
    oracle needs ~45 s per iteration here, so the run is checked through properties: the cost the
    engine reports equals the oracle's cost function evaluated on the returned state (initial and
    final), the cost is additive over point shards (two half-scene engines), it decreases
    monotonically, and the converged RMS sits at the injected noise level."""
    sc = ba.scenes.make_scene(**ba.scenes.CONFIGS["c3"])
    N, M = sc.n_points, sc.n_cams
    obs = O.ObsList(N, M, np.repeat(np.arange(N), M), np.tile(np.arange(M), N), sc.obs_xy, sc.obs_ptr)
    adj = ba.BundleAdjuster.from_observations(sc.obs_ptr, None, sc.obs_xy, sc.X0, sc.K0, sc.R0, sc.t0,
                                              f0=sc.f0, axis=sc.axis, dense=True)
    # initial cost: engine vs oracle on the normalised state, and additivity over two shards
    Xn, Rn, tn = O.normalize_gauge(sc.X0, sc.R0, sc.t0, sc.axis)
    f, u = sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy()
    E0 = adj.engine.cost(0)
    assert E0 == pytest.approx(O.cost(obs, Xn, f, u, Rn, tn, sc.f0), rel=1e-12)
    h = N // 2
    parts = []
    for lo, hi in ((0, h), (h, N)):
        eng = ba.Engine(hi - lo, M, (hi - lo) * M, sc.f0, sc.axis, True)
        eng.set_observations(None, None, sc.obs_xy[lo * M: hi * M])
        eng.set_state(Xn[lo:hi], Rn, tn, f, u)
        parts.append(eng.cost(0))
        eng.close()
    assert parts[0] + parts[1] == pytest.approx(E0, rel=1e-12)
    with contextlib.redirect_stdout(io.StringIO()):
        X, K, R, t = adj.optimize(2.0, 1e-8, max_iter=100)
    E = np.array([adj.records[0]["E_prev"]] + [r["E"] for r in adj.records])
    assert E[0] == pytest.approx(E0, rel=1e-13)
    assert np.all(np.diff(E) <= 0) and len(E) < 60
    rms = np.sqrt(E[-1] / sc.nobs)
    assert 0.9 * 0.005 * np.sqrt(2) < rms < 1.1 * 0.005 * np.sqrt(2)
    # the reported final cost is the oracle's cost of the returned state (gauge-invariant)
    Xf, Rf, tf = O.normalize_gauge(X, R, t, sc.axis)
    assert E[-1] == pytest.approx(O.cost(obs, Xf, K[:, 0, 0].copy(), K[:, :2, 2].copy(), Rf, tf, sc.f0), rel=1e-9)
    adj.engine.close()


def test_thousand_camera_sparse_run_properties(ba):
    """C4's shape at 1/50 of its points (1000 cameras x 20k points, 10 % visibility, n = 8993):
    the whole LM run on the sparse path (matrix-free pair kernel, two-level Cholesky, grid-wide
    back substitution).  Monotone cost, noise-level RMS, and the reported final cost equals the
    oracle's cost function on the returned state."""
    sc = ba.scenes.make_scene(1000, 20_000, seed=5, visibility=0.1)
    adj = ba.BundleAdjuster.from_observations(sc.obs_ptr, sc.obs_cam, sc.obs_xy, sc.X0, sc.K0, sc.R0, sc.t0,
                                              f0=sc.f0, axis=sc.axis, gauge_on_device=True)
    with contextlib.redirect_stdout(io.StringIO()):
        X, K, R, t = adj.optimize(2.0, 1e-8, max_iter=100)
    E = np.array([adj.records[0]["E_prev"]] + [r["E"] for r in adj.records])
    assert np.all(np.diff(E) <= 0) and 3 < len(E) < 60
    rms = np.sqrt(E[-1] / sc.nobs)
    assert 0.85 * 0.005 * np.sqrt(2) < rms < 1.1 * 0.005 * np.sqrt(2)
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr)),
                    sc.obs_cam.astype(np.int64), sc.obs_xy, sc.obs_ptr)
    Xf, Rf, tf = O.normalize_gauge(X, R, t, sc.axis)
    assert E[-1] == pytest.approx(O.cost(obs, Xf, K[:, 0, 0].copy(), K[:, :2, 2].copy(), Rf, tf, sc.f0), rel=1e-9)
    Xn, Rn, tn = O.normalize_gauge(sc.X0, sc.R0, sc.t0, sc.axis)
    assert E[0] == pytest.approx(O.cost(obs, Xn, sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy(), Rn, tn, sc.f0), rel=1e-11)
    adj.engine.close()


def test_shadow_module_intercepts_reference_import(ba):
    """`from lib.bundle_adjustment import BundleAdjuster` resolves to the B200 engine when the
    package directory precedes the reference checkout on sys.path (SURVEY.md section 8b)."""
    import importlib
    import sys

    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "lib" or k.startswith("lib.")}
    sys.path.insert(0, ba.PACKAGE_DIR)
    try:
        mod = importlib.import_module("lib.bundle_adjustment")
        assert mod.BundleAdjuster is ba.BundleAdjuster
    finally:
        sys.path.remove(ba.PACKAGE_DIR)
        for k in [k for k in sys.modules if k == "lib" or k.startswith("lib.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def _oracle_run(x, vis, X0, K0, R0, t0, axis, f0, max_iter):
    ora = O.OracleBundleAdjuster(x, X0, K0, R0, t0, f0=f0, visibility_index=vis, axis=axis)
    out = ora.optimize(2.0, 1e-8, max_iter=max_iter, verbose=False)
    return np.array([r["E"] for r in ora.trace]), out


def test_minimal_problem_two_cameras(ba):
    """Smallest admissible scene: 2 cameras (9 * 2 - 7 = 11 unknowns in one partial Cholesky panel),
    12 points; the whole run against the oracle."""
    sc = ba.scenes.make_scene(2, 12, seed=21, visibility=1.0)
    x, vis = sc.dense_x()
    adj = ba.BundleAdjuster(x, sc.X0, sc.K0, sc.R0, sc.t0, f0=sc.f0, axis=sc.axis)
    with contextlib.redirect_stdout(io.StringIO()):
        X, K, R, t = adj.optimize(2.0, 1e-8, max_iter=30)
    E = np.array([adj.records[0]["E_prev"]] + [r["E"] for r in adj.records])
    Eo, (Xo, Ko, Ro, to) = _oracle_run(x, None, sc.X0, sc.K0, sc.R0, sc.t0, sc.axis, sc.f0, 30)
    assert E.shape == Eo.shape
    np.testing.assert_allclose(E, Eo, rtol=1e-8)
    np.testing.assert_allclose(X, Xo, atol=1e-5)
    np.testing.assert_allclose(K, Ko, atol=1e-5)


def test_point_with_a_single_view_is_not_an_error(ba):
    """SURVEY.md 8b [probe]: a point seen once gives a rank-2 V_j that the reference does not
    detect (multiplicative damping makes it invertible); the run proceeds.  Same here, with the
    same first costs as the oracle."""
    g = load_golden("small_sparse_xup")
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    vis2 = vis.copy()
    vis2[5, :] = False
    vis2[5, 2] = True
    adj = ba.BundleAdjuster(x, X0, K0, R0, t0, visibility_index=vis2, axis=axis)
    with contextlib.redirect_stdout(io.StringIO()):
        adj.optimize(2.0, 1e-8, max_iter=3)
    E = np.array([adj.records[0]["E_prev"]] + [r["E"] for r in adj.records])
    Eo, _ = _oracle_run(x, vis2, X0, K0, R0, t0, axis, f0, 3)
    np.testing.assert_allclose(E, Eo[: len(E)], rtol=1e-7)


def test_retry_cap_raises_instead_of_looping_forever(ba):
    """Documented deviation (3): the reference's inner loop has no bound (:118).  Config 1's very
    first Gauss-Newton step is rejected (E 66.3 -> 3466 at c = 1e-4); with scale_factor = 1 the
    damping never grows, so the reference would repeat that solve forever.  The engine stops after
    max_retries solves with RuntimeError, and the state is left at the initial one."""
    g = load_golden("c1_euclid")
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    adj = ba.BundleAdjuster(x, X0, K0, R0, t0, visibility_index=vis, axis=axis, max_retries=5)
    with pytest.raises(RuntimeError, match="retries"):
        with contextlib.redirect_stdout(io.StringIO()):
            adj.optimize(1.0, 1e-8, max_iter=10)
    st = adj.engine.lm_state()
    assert st.count == 0 and st.solves == 5 and st.E == pytest.approx(float(g["E"][0]), rel=1e-9)


def test_c_abi_rejects_bad_arguments(ba):
    import ctypes as C

    cabi = ba.submodule("_cabi")
    lib = cabi.load()
    h = C.c_void_p()
    for kwargs in (dict(n_cams=1), dict(n_points=0), dict(axis=7), dict(f0=0.0), dict(device=99)):
        base = dict(n_points=10, n_obs=40, n_cams=4, axis=1, f0=1.0, dense=1, device=0)
        base.update(kwargs)
        if "n_points" in kwargs or "n_cams" in kwargs:
            base["n_obs"] = base["n_points"] * base["n_cams"]
        prob = cabi.Problem(base["n_points"], max(base["n_obs"], 0), base["n_cams"], base["axis"], base["f0"],
                            base["dense"], base["device"])
        assert lib.ba_create(C.byref(prob), C.byref(h)) == cabi.BA_ERR_INVALID
        assert lib.ba_last_error()
    # dense problem whose observation count does not match
    prob = cabi.Problem(10, 39, 4, 1, 1.0, 1, 0)
    assert lib.ba_create(C.byref(prob), C.byref(h)) == cabi.BA_ERR_INVALID
    # calls out of order
    eng = ba.Engine(10, 4, 40, 1.0, "x-up_z-forward", True)
    with pytest.raises(RuntimeError):
        eng.lm_begin(2.0, 1e-8, 10)
    eng.close()


def test_camera_without_observations_raises_like_the_reference(ba):
    """ADVICE r1: a camera nobody sees has an all-zero row in the reduced system.  The reference's
    LU raises LinAlgError("Singular matrix") on the first solve (:146); the Cholesky maps an
    exactly-zero pivot to the same error in the same solve instead of retrying 200 times."""
    g = load_golden("small_sparse_xup")
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    vis2 = vis.copy()
    vis2[:, 4] = False
    assert vis2.sum(axis=1).min() >= 2
    with pytest.raises(np.linalg.LinAlgError):
        _oracle_run(x, vis2, X0, K0, R0, t0, axis, f0, 3)
    adj = ba.BundleAdjuster(x, X0, K0, R0, t0, visibility_index=vis2, axis=axis)
    with pytest.raises(np.linalg.LinAlgError, match="Singular"):
        with contextlib.redirect_stdout(io.StringIO()):
            adj.optimize(2.0, 1e-8, max_iter=5)
    st = adj.engine.lm_state()
    assert st.solves == 1 and st.count == 0


def test_reference_constructor_takes_the_camera_major_block_as_it_lies_in_memory(ba):
    """Both reference scripts pass `np.stack(x_list).transpose(1, 0, 2)` (a camera-major block seen
    point-major, euclidiean_reconstruction.py:54).  The constructor uploads that block unchanged and
    re-orders it on the device (ba_set_observations_dense); the run is bit-identical to the one from
    a contiguous copy."""
    sc = ba.scenes.make_scene(37, 1234, seed=11)
    x, _ = sc.dense_x()
    xt = np.ascontiguousarray(x.transpose(1, 0, 2)).transpose(1, 0, 2)  # camera-major memory
    assert not xt.flags.c_contiguous and np.array_equal(xt, x)
    runs = []
    for arr in (x, xt, x.astype(np.float32).astype(np.float64)[:, :, ::1]):
        adj = ba.BundleAdjuster(arr, sc.X0, sc.K0, sc.R0, sc.t0, f0=sc.f0, axis=sc.axis)
        with contextlib.redirect_stdout(io.StringIO()):
            out = adj.optimize(2.0, 1e-8, max_iter=4)
        runs.append((np.array([r["E"] for r in adj.records]), out))
        adj.engine.close()
    assert np.array_equal(runs[0][0], runs[1][0])
    for a, b in zip(runs[0][1], runs[1][1]):
        assert np.array_equal(a, b)


def _fixture_run(ba, cfg, max_iter, tol):
    sc = ba.scenes.make_scene(**cfg)
    adj = ba.BundleAdjuster.from_observations(sc.obs_ptr, sc.obs_cam, sc.obs_xy, sc.X0, sc.K0, sc.R0, sc.t0,
                                              f0=sc.f0, axis=sc.axis)
    with contextlib.redirect_stdout(io.StringIO()):
        X, K, R, t = adj.optimize(2.0, tol, max_iter=max_iter)
    E = np.array([adj.records[0]["E_prev"]] + [r["E"] for r in adj.records])
    solves = np.array([0] + [r["solves"] for r in adj.records])
    adj.engine.close()
    return sc, E, solves, (X, K, R, t)


def test_thousand_camera_trajectory_matches_the_oracle(ba):
    """Config 4's shape (1000 cameras, 10 % visibility, n = 8993; 3000 points): ten LM iterations
    against the oracle's trajectory (tests/golden/c4_shape.npz, oracle/gen_golden_large.py) -- every
    accepted cost within 1e-9 relative, the same inner-solve count per iteration, the final state
    within 1e-6."""
    from oracle.gen_golden_large import C4_SHAPE

    g = load_golden("c4_shape")
    sc, E, solves, (X, K, R, t) = _fixture_run(ba, C4_SHAPE, 10, -1.0)
    assert sc.nobs == int(g["nobs"])
    assert E.shape == g["E"].shape
    np.testing.assert_allclose(E, g["E"], rtol=1e-9, atol=0)
    assert np.array_equal(solves, g["solves"])
    sub = int(g["sub"])
    np.testing.assert_allclose(X[::sub], g["X_sub"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(K, g["K"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(R, g["R"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(t, g["t"], rtol=0, atol=1e-6)


def test_global_camera_table_run_matches_the_oracle(ba):
    """1253 cameras (camera table in global memory, 177 64-blocks in the back substitution on at most
    148 CTAs), 10 % visibility: three LM iterations through the CUDA-graph loop against the oracle's
    (sparse Schur product, Cholesky solve) -- the bars of the thousand-camera trajectory.  Seed 1253:
    cond(S) = 1.1e5 at the initial state and c = 1e-4."""
    sc = ba.scenes.make_scene(1253, 2000, seed=1253, visibility=0.1)
    adj = ba.BundleAdjuster.from_observations(sc.obs_ptr, sc.obs_cam, sc.obs_xy, sc.X0, sc.K0, sc.R0, sc.t0,
                                              f0=sc.f0, axis=sc.axis)
    with contextlib.redirect_stdout(io.StringIO()):
        X, K, R, t = adj.optimize(2.0, -1.0, max_iter=3)
    E = np.array([adj.records[0]["E_prev"]] + [r["E"] for r in adj.records])
    solves = np.array([0] + [r["solves"] for r in adj.records])
    adj.engine.close()
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr)),
                    sc.obs_cam.astype(np.int64), sc.obs_xy, sc.obs_ptr)
    ora = O.OracleBundleAdjuster(None, sc.X0, sc.K0, sc.R0, sc.t0, f0=sc.f0, axis=sc.axis, obs=obs)
    Xo, Ko, Ro, to = ora.optimize(2.0, -1.0, max_iter=3, verbose=False, schur="sparse", solver="cholesky")
    assert len(E) == len(ora.trace) == 4
    np.testing.assert_allclose(E, [r["E"] for r in ora.trace], rtol=1e-9, atol=0)
    assert np.array_equal(solves, [r["solves"] for r in ora.trace])
    np.testing.assert_allclose(K, Ko, rtol=0, atol=1e-6)
    np.testing.assert_allclose(R, Ro, rtol=0, atol=1e-6)
    np.testing.assert_allclose(t, to, rtol=0, atol=1e-6)


def test_outlier_scene_converges_to_the_oracles_rms(ba):
    """Config 5's shape (1000 cameras, 10 % visibility, 1 % of the observations replaced by
    U[-0.5, 0.5]^2, plain L2 cost; 5000 points) run to convergence as BASELINE.json states it
    (optimize(2.0, 1e-8, max_iter=50)) against the CPU oracle's run on the same scene: the same
    number of accepted iterations, every cost within 1e-9 relative, the same converged RMS, the
    same final state."""
    from oracle.gen_golden_large import C5_SHAPE

    g = load_golden("c5_shape")
    sc, E, solves, (X, K, R, t) = _fixture_run(ba, C5_SHAPE, 50, 1e-8)
    assert sc.nobs == int(g["nobs"])
    assert E.shape == g["E"].shape, f"{len(E) - 1} accepted iterations, the oracle took {len(g['E']) - 1}"
    np.testing.assert_allclose(E, g["E"], rtol=1e-9, atol=0)
    assert np.array_equal(solves, g["solves"])
    rms = np.sqrt(E[-1] / sc.nobs)
    assert rms == pytest.approx(float(g["rms"]), rel=1e-9)
    assert rms > 3 * 0.005 * np.sqrt(2)  # the outliers dominate the converged error
    sub = int(g["sub"])
    np.testing.assert_allclose(X[::sub], g["X_sub"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(K, g["K"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(R, g["R"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(t, g["t"], rtol=0, atol=1e-6)


def test_unmodified_reference_script_runs_on_the_engine(ba, tmp_path):
    """BASELINE.json: "euclidiean_reconstruction.py runs it unchanged".  The byte-for-byte copy of
    the script under oracle/_ref (oracle/build_ref.py) is run through tools/run_reference_script.py:
    its self-calibration is the reference's own code, its BundleAdjuster resolves to this package.
    The printed iteration lines are compared with the ones the same script printed with the
    reference's own class (tests/golden/c1_euclid.npz)."""
    import os
    import subprocess
    import sys

    from oracle import build_ref

    if not build_ref.verify():
        pytest.skip("oracle/_ref not built (needs /root/reference at build time)")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = os.path.join(build_ref.REF_DST, "euclidiean_reconstruction.py")
    res = subprocess.run([sys.executable, os.path.join(root, "tools", "run_reference_script.py"), script],
                         capture_output=True, text=True, timeout=600,
                         env={**os.environ, "BA_SCRIPT_REPORT": str(tmp_path / "report.json")})
    assert res.returncode == 0, res.stderr[-2000:]
    got = [ln for ln in res.stdout.splitlines() if ln.startswith("Iteration ") and "reprojection_error_delta" in ln]
    ref = str(load_golden("c1_euclid")["stdout"]).strip().splitlines()
    # the initial value comes from the reference's SVD / eigen-decompositions on this host's BLAS:
    # same algorithm, last bits may differ from the build container's
    assert abs(len(got) - len(ref)) <= 2
    for a, b in list(zip(got, ref))[:10]:
        assert a.split(" = ")[0] == b.split(" = ")[0]
        assert float(a.split(" = ")[1]) == pytest.approx(float(b.split(" = ")[1]), rel=1e-5)
    import json

    rep = json.load(open(tmp_path / "report.json"))
    assert rep["adjuster_class"].endswith("bundle_adjuster.BundleAdjuster") and rep["kernel_launches"] > 0
