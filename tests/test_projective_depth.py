"""Projective-depth iteration, primary method (SURVEY.md section 8f row 3; reference
``lib/perspective_camera_calibration.py:61-144``): the oracle against the reference-generated
fixture (CPU), the CUDA path against both (GPU)."""
import contextlib
import io
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import depth_oracle as D  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "depth_primary.npz")
CASES = [("a", 200), ("b", 12)]


def _case(c):
    g = np.load(GOLDEN)
    return {k[2:]: g[k] for k in g.files if k.startswith(c + "_")}


@pytest.mark.parametrize("c,max_iter", CASES)
def test_oracle_matches_reference_fixture(c, max_iter):
    g = _case(c)
    x = D.create_data_matrix(list(g["xy"]), float(g["f0"]))
    assert np.array_equal(x, g["x"])  # _create_data_matrix (:35-41)
    z, errs = D.projective_depth_primary(x, float(g["f0"]), float(g["tol"]), max_iter)
    assert len(errs) == len(g["E"])
    np.testing.assert_allclose(z, g["z"], rtol=0, atol=1e-12)
    # the reference prints the error with 8 significant digits (:141); that is what the fixture holds
    np.testing.assert_allclose(errs, g["E"], rtol=2e-8)


def test_oracle_stops_at_the_tolerance():
    g = _case("a")
    z, errs = D.projective_depth_primary(g["x"], 1.0, 9.0e-3, 200)
    assert 1 < len(errs) < 200 and errs[-1] < 9.0e-3 <= errs[-2]


@pytest.mark.gpu
@pytest.mark.parametrize("c,max_iter", CASES)
def test_cuda_matches_reference_fixture_and_oracle(c, max_iter):
    import ba_b200

    g = _case(c)
    f0, tol = float(g["f0"]), float(g["tol"])
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        z = ba_b200.compute_projective_depth_primary_method(g["x"], f0, tol, max_iter)
    np.testing.assert_allclose(z, g["z"], rtol=0, atol=1e-9)
    lines = buf.getvalue().strip().splitlines()
    ref_lines = str(g["stdout"]).strip().splitlines()
    assert len(lines) == len(ref_lines)
    for a, b in zip(lines, ref_lines):
        if a.startswith("Iteration"):
            assert a.split("=")[0] == b.split("=")[0]
            assert float(a.split("=")[1]) == pytest.approx(float(b.split("=")[1]), rel=2e-8)
        else:
            assert a == b
    z2, errs = ba_b200.projective_depth_primary(g["x"], f0, tol, max_iter)
    assert np.array_equal(z2, z)  # bit-reproducible
    _, errs_o = D.projective_depth_primary(g["x"], f0, tol, max_iter)
    np.testing.assert_allclose(errs, errs_o, rtol=1e-10)


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,iters", [(40, 5000, 6), (3, 50, 4), (64, 700, 3)])
def test_cuda_matches_oracle_on_random_scenes(M, N, iters):
    """Wider Gram matrices (3M = 120, 192: several SYRK tiles, longer Jacobi sweeps), the minimum
    useful sizes, and early stopping."""
    import ba_b200

    sc = ba_b200.scenes.make_scene(M, N, seed=M + N, visibility=1.0)
    xd, _ = sc.dense_x()                      # (N, M, 2) image points
    x = np.concatenate((xd / sc.f0, np.ones((N, M, 1))), axis=2)
    z, errs = ba_b200.projective_depth_primary(x, sc.f0, 1e-12, iters)
    zo, errs_o = D.projective_depth_primary(x, sc.f0, 1e-12, iters)
    assert len(errs) == iters
    np.testing.assert_allclose(errs, errs_o, rtol=1e-9)
    np.testing.assert_allclose(z, zo, rtol=0, atol=1e-9 * np.abs(zo).max())
    # stops as soon as the tolerance is met
    z1, e1 = ba_b200.projective_depth_primary(x, sc.f0, errs_o[1] * 1.0000001, iters)
    assert len(e1) == 2


@pytest.mark.gpu
def test_cuda_rejects_bad_shapes():
    import ba_b200

    with pytest.raises(ValueError):
        ba_b200.projective_depth_primary(np.ones((10, 3, 2)), 1.0, 1e-3)
    with pytest.raises(ValueError):
        ba_b200.projective_depth_primary(np.ones((10, 65, 3)), 1.0, 1e-3)


@pytest.mark.gpu
def test_shadow_module_swaps_the_primary_method(tmp_path):
    """`from lib.perspective_camera_calibration import ...` behind the package directory keeps the
    next module's code and replaces only the primary depth iteration (checked with a stand-in for the
    reference checkout, which does not exist on the GPU box)."""
    import importlib

    import ba_b200

    ref = tmp_path / "ref" / "lib"
    ref.mkdir(parents=True)
    (ref / "perspective_camera_calibration.py").write_text(
        "def _compute_projective_depth_primary_method(x, f0, tolerance, max_iter=200):\n    return 'reference'\n"
        "def perspective_self_calibration(x, f0=1.0, tol=0.01, method='primary'):\n"
        "    return _compute_projective_depth_primary_method(x, f0, tol)\n"
        "def untouched():\n    return 'kept'\n")
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "lib" or k.startswith("lib.")}
    sys.path[:0] = [ba_b200.PACKAGE_DIR, str(tmp_path / "ref")]
    try:
        mod = importlib.import_module("lib.perspective_camera_calibration")
        assert mod.untouched() == "kept"
        g = _case("b")
        with contextlib.redirect_stdout(io.StringIO()):
            z = mod.perspective_self_calibration(g["x"], float(g["f0"]), 5.47e-3)
        assert isinstance(z, np.ndarray) and z.shape == g["z"].shape
    finally:
        sys.path.remove(ba_b200.PACKAGE_DIR)
        sys.path.remove(str(tmp_path / "ref"))
        for k in [k for k in sys.modules if k == "lib" or k.startswith("lib.")]:
            del sys.modules[k]
        sys.modules.update(saved)


# ---- dual method (reference :147-235) and the rank-4 factorisation (lib/factorization.py) ----------
def test_dual_oracle_matches_reference_fixture_up_to_a_sign_per_image():
    """The dual method's per-image eigenvector signs are LAPACK's choice (the reference's sign rule
    flips rows, :212-215, not the per-image columns), and the reference's own Euclidean upgrade is
    invariant to them (asserted when the fixture is generated, ``oracle/gen_golden_depth_dual.py``).
    The restatement (rank-12 factorisation of the N x N eigenproblems) reproduces the reference's
    depths up to that sign: the script's one pass (tol 1e-2, ``euclidiean_reconstruction.py:42``) and
    a 15-pass run."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "depth_dual.npz"))
    for zkey, ekey, tol, iters in (("z", "E", float(g["tol"]), 50), ("z15", "E15", 1e-9, 15)):
        z, errs = D.projective_depth_dual(g["x"], float(g["f0"]), tol, iters)
        assert len(errs) == len(g[ekey])
        sign = np.sign((z * g[zkey]).sum(axis=0))
        assert set(np.unique(sign)) <= {-1.0, 1.0}
        np.testing.assert_allclose(z * sign, g[zkey], rtol=0, atol=1e-11)
        np.testing.assert_allclose(errs, g[ekey], rtol=2e-8)


DUAL = os.path.join(ROOT, "tests", "golden", "depth_dual.npz")


@pytest.mark.gpu
def test_cuda_dual_method_matches_oracle_and_reference_fixture():
    """The CUDA dual method against the oracle (same per-image sign rule: exact comparison) and
    against the unmodified reference's depths (up to the sign per image that LAPACK chose there)."""
    import ba_b200

    g = np.load(DUAL)
    f0 = float(g["f0"])
    for zkey, ekey, tol, iters in (("z", "E", float(g["tol"]), 50), ("z15", "E15", 1e-9, 15)):
        z, errs = ba_b200.projective_depth_dual(g["x"], f0, tol, iters)
        zo, errs_o = D.projective_depth_dual(g["x"], f0, tol, iters)
        assert len(errs) == len(errs_o) == len(g[ekey])
        np.testing.assert_allclose(errs, errs_o, rtol=1e-10)
        np.testing.assert_allclose(z, zo, rtol=0, atol=1e-9 * np.abs(zo).max())
        sign = np.sign((z * g[zkey]).sum(axis=0))
        np.testing.assert_allclose(z * sign, g[zkey], rtol=0, atol=1e-9)
        np.testing.assert_allclose(errs, g[ekey], rtol=2e-8)
    z2, _ = ba_b200.projective_depth_dual(g["x"], f0, 1e-9, 15)
    assert np.array_equal(z2, z)  # bit-reproducible
    # printed lines of the reference signature (:227-233)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        ba_b200.compute_projective_depth_dual_method(g["x"], f0, float(g["tol"]))
    assert buf.getvalue().strip() == f"Iteration 1: reprojection_error = {float(g['E'][0]):.8}"


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,iters", [(40, 3000, 4), (3, 40, 3), (64, 500, 2), (33, 257, 3)])
def test_cuda_dual_method_matches_oracle_on_random_scenes(M, N, iters):
    import ba_b200

    sc = ba_b200.scenes.make_scene(M, N, seed=M + N, visibility=1.0)
    xd, _ = sc.dense_x()
    x = np.concatenate((xd / sc.f0, np.ones((N, M, 1))), axis=2)
    z, errs = ba_b200.projective_depth_dual(x, sc.f0, 1e-12, iters)
    zo, errs_o = D.projective_depth_dual(x, sc.f0, 1e-12, iters)
    assert len(errs) == iters
    np.testing.assert_allclose(errs, errs_o, rtol=1e-9)
    np.testing.assert_allclose(z, zo, rtol=0, atol=1e-9 * np.abs(zo).max())
    # max_iter < 1 runs one pass, like the reference's loop (:162-231)
    _, e0 = ba_b200.projective_depth_dual(x, sc.f0, 1e-12, 0)
    assert len(e0) == 1


@pytest.mark.gpu
@pytest.mark.parametrize("M,N", [(10, 200), (40, 3000), (2, 9), (64, 1000)])
def test_cuda_factorisation_matches_lapack_svd(M, N):
    """factorization_method (lib/factorization.py:5-15): M = U[:, :4], S = diag(Sigma[:4]) Vt[:4],
    singular vectors up to sign; the product M S is unique."""
    import ba_b200

    rs = np.random.RandomState(M * 1000 + N)
    # a rank-4 matrix plus noise, like the scaled observation matrix of the perspective pipeline
    W = rs.standard_normal((3 * M, 4)) @ rs.standard_normal((4, N)) + 1e-3 * rs.standard_normal((3 * M, N))
    Mg, Sg, sg = ba_b200.factorize_rank4(W)
    U, Sigma, Vt = np.linalg.svd(W, full_matrices=False)
    np.testing.assert_allclose(sg, Sigma[:4], rtol=1e-10)
    sign = np.sign((Mg * U[:, :4]).sum(axis=0))
    np.testing.assert_allclose(Mg * sign, U[:, :4], rtol=0, atol=1e-9)
    np.testing.assert_allclose(Sg * sign[:, None], Sigma[:4, None] * Vt[:4], rtol=0, atol=1e-9 * Sigma[0])
    np.testing.assert_allclose(Mg @ Sg, (U[:, :4] * Sigma[:4]) @ Vt[:4], rtol=0, atol=1e-9 * Sigma[0])
    np.testing.assert_allclose(Mg.T @ Mg, np.eye(4), rtol=0, atol=1e-12)


@pytest.mark.gpu
def test_jacobi_fallback_matches_reference_fixture(monkeypatch):
    """The eigenspace normally comes from a warm-started subspace iteration; the parallel Jacobi
    solver behind it (near-degenerate spectra) is forced here through its switch, which every call
    reads, and has to meet the bars of each entry point's default-path test: the primary method on
    fixture b, the dual method on its fixture, the factorisation on one of the LAPACK cases."""
    monkeypatch.setenv("BA_DEPTH_JACOBI", "1")
    test_cuda_matches_reference_fixture_and_oracle("b", 12)
    test_cuda_dual_method_matches_oracle_and_reference_fixture()
    test_cuda_factorisation_matches_lapack_svd(40, 3000)


@pytest.mark.gpu
def test_shadowed_self_calibration_reproduces_the_reference_on_the_scripts_scene():
    """SURVEY.md 8f row 3, VERDICT r1 item 8: `perspective_self_calibration(x_list, 1.0, tol=1e-2,
    method="dual")` (euclidiean_reconstruction.py:42) through the shadow module -- dual depths and
    the rank-4 factorisation on the GPU, the reference's own Euclidean upgrade on top -- against what
    the unmodified reference returned for the same scene (tests/golden/depth_dual.npz): (X, R, t, K)
    within 1e-9.  The reference's code comes from the build-time copy oracle/_ref."""
    import importlib

    import ba_b200
    from oracle import build_ref

    if not build_ref.verify():
        pytest.skip("oracle/_ref not built (needs /root/reference at build time)")
    g = np.load(DUAL)
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "lib" or k.startswith("lib.")}
    sys.path[:0] = [ba_b200.PACKAGE_DIR, build_ref.REF_DST]
    launches0 = ba_b200.submodule("engine").launch_count()
    try:
        mod = importlib.import_module("lib.perspective_camera_calibration")
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            X, R, t, K = mod.perspective_self_calibration(list(g["xy"]), 1.0, tol=1e-2, method="dual")
        assert buf.getvalue().startswith("Iteration 1: reprojection_error = ")
        assert ba_b200.submodule("engine").launch_count() > launches0  # the GPU stages ran
        for got, name in ((X, "X"), (R, "R"), (t, "t"), (K, "K")):
            np.testing.assert_allclose(got, g[name], rtol=0, atol=1e-9 * max(1.0, np.abs(g[name]).max()), err_msg=name)
        # more images than the kernels take: the reference's own code runs instead
        xbig = np.ones((8, 70, 3))
        assert mod._compute_projective_depth_dual_method.__module__.endswith("perspective_camera_calibration")
        assert not mod._fits(xbig)
    finally:
        sys.path.remove(ba_b200.PACKAGE_DIR)
        sys.path.remove(build_ref.REF_DST)
        for k in [k for k in sys.modules if k == "lib" or k.startswith("lib.")]:
            del sys.modules[k]
        sys.modules.update(saved)
