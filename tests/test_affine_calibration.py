"""Affine self-calibrations (SURVEY.md section 8f row 4; reference
``lib/affine_camera_calibration.py:7, :59, :137``).

CPU: the oracle restatement against the reference-generated fixture (all eight sign choices of the
three singular vectors), and the product's host-side O(M) algebra against the same fixture when it
is fed a LAPACK factorisation.  GPU: the whole path -- centred rank-4 factorisation on the tensor
cores + host algebra -- against the unmodified reference's outputs.

Parity bar: 1e-9 absolute on S (scene scale ~1) and R.  The reference's answer depends on the signs
LAPACK returns for the singular vectors; the GPU path fixes them by its own rule, so the comparison
first reads the relative signs off the factorisation and then requires the match for EVERY one of
the eight classes (``signs=``), i.e. also for the mirror solutions."""
import importlib
import itertools
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import affine_oracle as AO  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "affine_calib.npz")
MODELS = ("orthographic", "symmetric_affine", "paraperspective")
CASES = ("script", "wide")
SIGNS = list(itertools.product((1.0, -1.0), repeat=3))


def _tag(d):
    return "".join("p" if v > 0 else "m" for v in d)


def _data(g, case):
    return [x.copy() for x in g[f"{case}_xy"]], g[f"{case}_f"]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("model", MODELS)
def test_oracle_matches_reference_fixture(case, model):
    g = np.load(GOLDEN)
    xl, f = _data(g, case)
    S, R = AO.self_calibration(model, xl, f)
    np.testing.assert_allclose(S, g[f"{case}_{model}_S"], rtol=0, atol=1e-11)
    np.testing.assert_allclose(R, g[f"{case}_{model}_R"], rtol=0, atol=1e-11)
    for d in SIGNS:
        S, R = AO.self_calibration(model, xl, f, signs=d)
        np.testing.assert_allclose(S, g[f"{case}_{model}_S_{_tag(d)}"], rtol=0, atol=1e-11)
        np.testing.assert_allclose(R, g[f"{case}_{model}_R_{_tag(d)}"], rtol=0, atol=1e-11)


def test_fixture_sign_classes_are_what_the_docstring_says():
    """det D = +1: a half-turn of the world frame, (S D, D R); det D = -1: a different (mirror) answer."""
    g = np.load(GOLDEN)
    for case in CASES:
        S, R = g[f"{case}_paraperspective_S"], g[f"{case}_paraperspective_R"]
        d = np.array([1.0, -1.0, -1.0])
        np.testing.assert_allclose(g[f"{case}_paraperspective_S_pmm"], S * d, atol=1e-10)
        np.testing.assert_allclose(g[f"{case}_paraperspective_R_pmm"], d[None, :, None] * R, atol=1e-10)
        m = np.array([1.0, 1.0, -1.0])
        assert np.abs(g[f"{case}_paraperspective_R_ppm"] - m[None, :, None] * R).max() > 1e-3


def _lapack_factors(xl):
    W = np.hstack(xl).T.copy()
    t = W.mean(axis=1)
    Wc = W - t[:, None]
    U, s, Vt = np.linalg.svd(Wc, full_matrices=False)
    return U[:, :3], s[:3, None] * Vt[:3], t.reshape(-1, 2)


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("model", MODELS)
def test_host_algebra_matches_reference_fixture(case, model):
    """calibrate_from_factors (the product's O(M) NumPy stage, written on 6-vectors) fed LAPACK's
    factors reproduces the unmodified reference for every sign class."""
    import ba_b200

    ac = ba_b200.submodule("affine_calibration")
    g = np.load(GOLDEN)
    xl, f = _data(g, case)
    U3, S3, t = _lapack_factors(xl)
    for d in SIGNS:
        S, R = ac.calibrate_from_factors(model, U3, S3, t, f, signs=d)
        np.testing.assert_allclose(S, g[f"{case}_{model}_S_{_tag(d)}"], rtol=0, atol=1e-10)
        np.testing.assert_allclose(R, g[f"{case}_{model}_R_{_tag(d)}"], rtol=0, atol=1e-10)


def test_host_algebra_error_behaviour():
    import ba_b200

    ac = ba_b200.submodule("affine_calibration")
    g = np.load(GOLDEN)
    xl, f = _data(g, "wide")
    U3, S3, t = _lapack_factors(xl)
    with pytest.raises(ValueError):
        ac.calibrate_from_factors("perspective", U3, S3, t, f)
    with pytest.raises(ValueError):          # reference :145-146
        ac.paraperspective_self_calibration(xl, f[:-1])
    with pytest.raises(ValueError):          # reference :232-234 (ragged input)
        ac.orthographic_self_calibration(xl[:-1] + [xl[-1][:-1]])
    U3c, S3c = ac.canonical_signs(-U3, -S3)
    pick = np.abs(U3c).argmax(axis=0)
    assert (U3c[pick, np.arange(3)] > 0).all()
    np.testing.assert_allclose(U3c @ S3c, U3 @ S3, atol=1e-12)


def _relative_signs(ac, xl):
    """d with U_lapack = U_gpu d (per column), from the GPU factorisation itself."""
    U3g, S3g, sig, t = ac.factorize_observations(xl)
    U3l, S3l, tl = _lapack_factors(xl)
    d = np.sign(np.sum(U3l * U3g, axis=0))
    return d, (U3g, S3g, sig, t), (U3l, S3l, tl)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_cuda_centred_factorisation_matches_lapack(case):
    import ba_b200

    ac = ba_b200.submodule("affine_calibration")
    g = np.load(GOLDEN)
    xl, _ = _data(g, case)
    d, (U3g, S3g, sig, t), (U3l, S3l, tl) = _relative_signs(ac, xl)
    np.testing.assert_allclose(t, tl, rtol=0, atol=1e-14)
    np.testing.assert_allclose(U3g * d[None, :], U3l, rtol=0, atol=1e-10)
    np.testing.assert_allclose(S3g * d[:, None], S3l, rtol=0, atol=1e-10 * np.abs(S3l).max())
    np.testing.assert_allclose(sig, np.linalg.norm(S3l, axis=1), rtol=1e-11)
    pick = np.abs(U3g).argmax(axis=0)
    assert (U3g[pick, np.arange(3)] > 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("model", MODELS)
def test_cuda_self_calibration_matches_reference_fixture(case, model):
    import ba_b200

    ac = ba_b200.submodule("affine_calibration")
    g = np.load(GOLDEN)
    xl, f = _data(g, case)
    d_rel, _, _ = _relative_signs(ac, xl)
    fn = getattr(ba_b200, f"{model}_self_calibration")
    launches0 = ba_b200.submodule("engine").launch_count()
    for d in SIGNS:
        args = (xl, f) if model == "paraperspective" else (xl,)
        S, R = fn(*args, signs=d)
        ref = _tag(np.array(d) * d_rel)     # the LAPACK sign class this choice corresponds to
        np.testing.assert_allclose(S, g[f"{case}_{model}_S_{ref}"], rtol=0, atol=1e-9)
        np.testing.assert_allclose(R, g[f"{case}_{model}_R_{ref}"], rtol=0, atol=1e-9)
    assert ba_b200.submodule("engine").launch_count() > launches0
    # bit-reproducible
    args = (xl, f) if model == "paraperspective" else (xl,)
    S1, R1 = fn(*args)
    S2, R2 = fn(*args)
    assert np.array_equal(S1, S2) and np.array_equal(R1, R2)


@pytest.mark.gpu
def test_cuda_self_calibration_at_a_size_the_reference_cannot_hold():
    """60 images x 200 000 points: the reference's full SVD would need a 320 GB factor.  Properties:
    rank-3 reproduction of the centred observations at the noise level, orthogonal rotations, and
    agreement with a LAPACK factorisation of the small Gram matrix."""
    import ba_b200

    ac = ba_b200.submodule("affine_calibration")
    rng = np.random.default_rng(11)
    M, N = 60, 200_000
    X = rng.normal(0, 1.0, (N, 3))
    xl = []
    for i in range(M):
        q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        c = q.T @ X.T
        xl.append((c[:2] / (40.0 + c[2])).T + rng.normal(0, 0.05, 2) + 1e-4 * rng.normal(size=(N, 2)))
    U3, S3, sig, t = ac.factorize_observations(xl)
    W = np.hstack(xl).T
    Wc = W - W.mean(axis=1)[:, None]
    np.testing.assert_allclose(t.ravel(), W.mean(axis=1), rtol=0, atol=1e-13)
    lam, vec = np.linalg.eigh(Wc @ Wc.T)
    np.testing.assert_allclose(sig, np.sqrt(lam[::-1][:3]), rtol=1e-10)
    proj = vec[:, ::-1][:, :3]
    np.testing.assert_allclose(U3 @ U3.T, proj @ proj.T, rtol=0, atol=1e-8)
    resid = Wc - U3 @ S3
    assert np.sqrt(np.mean(resid ** 2)) < 2.0 * np.sqrt(np.mean((Wc - proj @ (proj.T @ Wc)) ** 2)) + 1e-12
    S, R = ba_b200.paraperspective_self_calibration(xl, 40.0 * np.ones(M))
    assert S.shape == (N, 3) and R.shape == (M, 3, 3)
    np.testing.assert_allclose(np.einsum("nij,nkj->nik", R, R), np.broadcast_to(np.eye(3), (M, 3, 3)), atol=1e-12)


@pytest.mark.gpu
def test_shadow_module_runs_the_scripts_call_on_the_gpu(tmp_path):
    """`from lib.affine_camera_calibration import paraperspective_self_calibration`
    (affine_reconstruction.py:3-7, :42) behind the package directory, against what the unmodified
    reference returned; the next module on sys.path is a stand-in for the reference's, since the
    call the script makes never reaches it."""
    import ba_b200

    ref_dir = tmp_path / "ref"
    (ref_dir / "lib").mkdir(parents=True)
    (ref_dir / "lib" / "affine_camera_calibration.py").write_text(
        "def orthographic_self_calibration(data_list):\n    return 'reference'\n"
        "def symmetric_affine_self_calibration(data_list):\n    return 'reference'\n"
        "def paraperspective_self_calibration(data_list, f):\n    return 'reference'\n"
        "def _get_T(tau):\n    return 'kept'\n")
    g = np.load(GOLDEN)
    xl, f = _data(g, "script")
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "lib" or k.startswith("lib.")}
    sys.path[:0] = [ba_b200.PACKAGE_DIR, str(ref_dir)]
    launches0 = ba_b200.submodule("engine").launch_count()
    try:
        mod = importlib.import_module("lib.affine_camera_calibration")
        S, R = mod.paraperspective_self_calibration(xl, f)
        assert ba_b200.submodule("engine").launch_count() > launches0
        ac = ba_b200.submodule("affine_calibration")
        d_rel, _, _ = _relative_signs(ac, xl)
        ref = _tag(d_rel)
        np.testing.assert_allclose(S, g[f"script_paraperspective_S_{ref}"], rtol=0, atol=1e-9)
        np.testing.assert_allclose(R, g[f"script_paraperspective_R_{ref}"], rtol=0, atol=1e-9)
        assert mod._get_T is sys.modules["lib._reference_affine_camera_calibration"]._get_T
        # more images than the kernels take: the reference's own function answers
        assert not mod._fits([np.zeros((10, 2))] * 70)
    finally:
        sys.path.remove(ba_b200.PACKAGE_DIR)
        sys.path.remove(str(ref_dir))
        for k in [k for k in sys.modules if k == "lib" or k.startswith("lib.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_shadow_module_falls_through_for_inputs_the_kernels_do_not_take(tmp_path):
    """CPU: with a stand-in for the reference checkout, an input with more than 64 images goes to the
    next module's function; other names are the next module's."""
    import ba_b200

    ref = tmp_path / "ref" / "lib"
    ref.mkdir(parents=True)
    (ref / "affine_camera_calibration.py").write_text(
        "def orthographic_self_calibration(data_list):\n    return 'reference'\n"
        "def symmetric_affine_self_calibration(data_list):\n    return 'reference'\n"
        "def paraperspective_self_calibration(data_list, f):\n    return 'reference'\n"
        "def _get_T(tau):\n    return 'kept'\n")
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "lib" or k.startswith("lib.")}
    sys.path[:0] = [ba_b200.PACKAGE_DIR, str(tmp_path / "ref")]
    try:
        mod = importlib.import_module("lib.affine_camera_calibration")
        many = [np.zeros((10, 2))] * 70
        assert mod.orthographic_self_calibration(many) == "reference"
        assert mod.paraperspective_self_calibration(many, np.ones(70)) == "reference"
        assert mod._get_T(None) == "kept"
    finally:
        sys.path.remove(ba_b200.PACKAGE_DIR)
        sys.path.remove(str(tmp_path / "ref"))
        for k in [k for k in sys.modules if k == "lib" or k.startswith("lib.")]:
            del sys.modules[k]
        sys.modules.update(saved)
