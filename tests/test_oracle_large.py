"""CPU checks of the oracle's large-configuration legs: the sparsity-aware C restatement of the Schur
reduction against the dense NumPy form (which the reference's golden vectors pin), the oracle at the
full config 2 against two iterations of the UNMODIFIED reference (tests/golden/c2_reference.npz,
oracle/gen_golden_large.py), and the build-time copy of the reference (oracle/_ref)."""

import numpy as np
import pytest

import ba_b200
from conftest import case_inputs, load_golden
from oracle import ba_oracle as O
from oracle import build_ref


def _obs(sc):
    return O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr)),
                     sc.obs_cam.astype(np.int64), sc.obs_xy, sc.obs_ptr)


@pytest.mark.parametrize("n_cams,n_points,vis", [(12, 300, 0.5), (40, 500, 0.2), (7, 50, 1.0), (33, 64, 0.1)])
def test_sparse_schur_restatement_equals_dense_form(n_cams, n_points, vis):
    sc = ba_b200.scenes.make_scene(n_cams, n_points, seed=n_cams, visibility=vis)
    obs = _obs(sc)
    X, R, t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, sc.axis)
    f, u = sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy()
    lin = O.linearize(obs, X, f, u, R, t, sc.f0)
    A1, b1, V1 = O.reduced_system(obs, lin, 1e-3)
    A2, b2, V2 = O.reduced_system_sparse(obs, lin, 1e-3)
    np.testing.assert_allclose(A2, A1, rtol=0, atol=1e-13 * np.abs(A1).max())
    np.testing.assert_allclose(b2, b1, rtol=0, atol=1e-13 * np.abs(b1).max())
    # off-diagonal camera blocks are mirrored exactly; a diagonal block is W^T V^-1 W evaluated entry
    # by entry, symmetric to rounding
    np.testing.assert_allclose(A2, A2.T, rtol=0, atol=1e-14 * np.abs(A1).max())
    off = np.kron(1 - np.eye(n_cams), np.ones((9, 9))).astype(bool)
    assert np.array_equal(A2[off], A2.T[off])
    assert np.array_equal(V1, V2)
    m = np.diff(obs.ptr)
    assert O.schur_flops_sparse(obs) == pytest.approx(float(np.sum(3.0 * 9 * m * (9 * m + 1))))


def test_sparse_cholesky_run_equals_dense_lu_run_on_a_reference_golden_case():
    g = load_golden("small_sparse_xup")
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    ora = O.OracleBundleAdjuster(x, X0, K0, R0, t0, f0=f0, visibility_index=vis, axis=axis)
    X, K, R, t = ora.optimize(2.0, 1e-8, max_iter=100, verbose=False, schur="sparse", solver="cholesky")
    E = np.array([r["E"] for r in ora.trace])
    assert E.shape == g["E"].shape
    np.testing.assert_allclose(E, g["E"], rtol=1e-9)
    np.testing.assert_allclose(X, g["X"], atol=1e-6)
    np.testing.assert_allclose(K, g["K"], atol=1e-6)


def test_oracle_matches_reference_at_c2():
    """BASELINE.md section 3.3: the oracle is trusted at C3-C5 only if it matches the true reference at
    C2 too.  Two iterations of the unmodified reference at the full config 2 were recorded in the
    build container (16 GB, ~20 s per iteration); the oracle replays them here in seconds."""
    g = load_golden("c2_reference")
    sc = ba_b200.scenes.make_scene(**ba_b200.scenes.CONFIGS["c2"])
    ora = O.OracleBundleAdjuster(None, sc.X0, sc.K0, sc.R0, sc.t0, f0=sc.f0, axis=sc.axis, obs=_obs(sc))
    X, K, R, t = ora.optimize(2.0, 1e-8, max_iter=2, verbose=False)
    E = np.array([r["E"] for r in ora.trace])
    np.testing.assert_allclose(E, g["E"], rtol=1e-11)
    sub = int(g["sub"])
    np.testing.assert_allclose(X[::sub], g["X_sub"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(X.sum(axis=0), g["X_sum"], rtol=0, atol=1e-7)
    np.testing.assert_allclose(K, g["K"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(R, g["R"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(t, g["t"], rtol=0, atol=1e-9)


def test_chunk_seeded_scene_shards_tile_the_whole_scene():
    cfg = dict(n_cams=9, n_points=5000, seed=8, visibility=0.4, outlier_frac=0.02, chunk_seeded=True, chunk=700)
    whole = ba_b200.scenes.make_scene(**cfg)
    world = 3
    for r in range(world):
        lo, hi = cfg["n_points"] * r // world, cfg["n_points"] * (r + 1) // world
        part = ba_b200.scenes.make_scene(**cfg, point_range=(lo, hi))
        a, b = whole.obs_ptr[lo], whole.obs_ptr[hi]
        assert np.array_equal(part.obs_xy, whole.obs_xy[a:b]) and np.array_equal(part.obs_cam, whole.obs_cam[a:b])
        assert np.array_equal(part.obs_ptr, whole.obs_ptr[lo:hi + 1] - a)
        assert np.array_equal(part.X0, whole.X0[lo:hi]) and np.array_equal(part.R0, whole.R0)
    with pytest.raises(ValueError):
        ba_b200.scenes.make_scene(9, 100, point_range=(0, 10))


def _stand_in_reference(root):
    """A reference checkout in miniature: the lib/ modules load_reference_class() imports and a script."""
    (root / "lib").mkdir(parents=True)
    (root / "lib" / "utils.py").write_text("def unit_vec(v):\n    return v\n")
    (root / "lib" / "bundle_adjustment.py").write_text(
        "from lib.utils import unit_vec\n\n\nclass BundleAdjuster:\n    def __init__(self, x):\n        self.x = unit_vec(x)\n")
    (root / "euclidiean_reconstruction.py").write_text("print('script')\n")
    return root


def test_oracle_ref_is_a_byte_for_byte_copy_of_the_reference(tmp_path, monkeypatch):
    src = _stand_in_reference(tmp_path / "reference")
    dst = tmp_path / "_ref"
    monkeypatch.setattr(build_ref, "REF_SRC", str(src))
    monkeypatch.setattr(build_ref, "REF_DST", str(dst))
    build_ref.build()
    assert build_ref.verify()
    for name in ["lib/utils.py", "lib/bundle_adjustment.py", "euclidiean_reconstruction.py"]:
        assert (src / name).read_bytes() == (dst / name).read_bytes()
    # the class bench.py times is the reference's own, not the product's
    cls = build_ref.load_reference_class()
    assert cls.__module__ == "lib.bundle_adjustment" and cls.__init__.__code__.co_filename.startswith(str(dst))
    assert cls is not ba_b200.BundleAdjuster and cls("x").x == "x"


def test_reference_copy_detects_modification(tmp_path, monkeypatch):
    dst = tmp_path / "_ref"
    monkeypatch.setattr(build_ref, "REF_SRC", str(_stand_in_reference(tmp_path / "reference")))
    monkeypatch.setattr(build_ref, "REF_DST", str(dst))
    build_ref.build()
    assert build_ref.verify()
    with open(dst / "lib" / "utils.py", "a") as f:
        f.write("\n# edited\n")
    assert not build_ref.verify()
    with pytest.raises(RuntimeError):
        build_ref.load_reference_class()
