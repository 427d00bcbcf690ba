"""Batched re-projection (`calc_projected_points`, reference lib/camera.py:74-81): the oracle
restatement against a fixture produced by the unmodified reference, and the CUDA kernel (through
`ba_project_points` of the C ABI) against the oracle."""
import os

import numpy as np
import pytest

from oracle import ba_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "projection.npz")


def test_oracle_projection_matches_reference_fixture():
    g = np.load(GOLDEN)
    x = O.project_all(g["X"], g["K"], g["R"], g["t"])
    assert x.shape == g["x"].shape
    np.testing.assert_allclose(x, g["x"], rtol=1e-13, atol=1e-14)


def test_oracle_projection_agrees_with_ba_projection():
    """For K = [[f,0,u0],[0,f,v0],[0,0,f0]] it is the projection the BA cost uses (:299-305)."""
    import ba_b200

    sc = ba_b200.scenes.make_scene(6, 40, seed=3)
    x = O.project_all(sc.X0, sc.K0, sc.R0, sc.t0)
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), sc.n_cams),
                    np.tile(np.arange(sc.n_cams), sc.n_points), sc.obs_xy, sc.obs_ptr)
    p, q, r = O.project(obs, sc.X0, sc.K0[:, 0, 0], sc.K0[:, :2, 2], sc.R0, sc.t0, sc.f0)[:3]
    ref = np.stack([p / r, q / r], axis=1).reshape(sc.n_points, sc.n_cams, 2).transpose(1, 0, 2)
    np.testing.assert_allclose(x, ref, rtol=1e-12, atol=1e-13)


@pytest.mark.gpu
@pytest.mark.parametrize("M,N", [(9, 157), (1, 1), (3, 70001), (130, 515)])
def test_cuda_projection_matches_oracle(M, N):
    import ba_b200

    if (M, N) == (9, 157):
        g = np.load(GOLDEN)
        X, K, R, t = g["X"], g["K"], g["R"], g["t"]
    else:
        sc = ba_b200.scenes.make_scene(max(M, 2), N, seed=M)
        rng = np.random.RandomState(N)
        X, K, R, t = sc.X0, sc.K0[:M] + rng.normal(0, 0.01, (M, 3, 3)), sc.R0[:M], sc.t0[:M]
    got = ba_b200.calc_projected_points(X, K, R, t)
    assert isinstance(got, list) and len(got) == M and got[0].shape == (N, 2)
    want = O.project_all(X, K, R, t)
    np.testing.assert_allclose(np.stack(got), want, rtol=1e-12, atol=1e-13)


@pytest.mark.gpu
def test_cuda_projection_rejects_bad_shapes():
    import ba_b200

    with pytest.raises(ValueError):
        ba_b200.calc_projected_points(np.zeros((4, 2)), np.zeros((2, 3, 3)), np.zeros((2, 3, 3)), np.zeros((2, 3)))


def test_shadow_camera_module_keeps_reference_code_and_swaps_projection(tmp_path):
    """With this package's directory before the reference on sys.path, `lib.camera` is the
    reference's module except for `calc_projected_points` (SURVEY.md section 8b / 8f); checked with a
    stand-in for the reference's lib/camera.py, whose names and module-internal calls must survive."""
    import importlib
    import sys

    import ba_b200

    ref = tmp_path / "ref" / "lib"
    ref.mkdir(parents=True)
    (ref / "camera.py").write_text(
        "class Camera:\n"
        "    @staticmethod\n"
        "    def create(pos, target, f=1, f0=1):\n        return 'reference camera'\n"
        "def calc_projected_points(X, K, R, t):\n    return 'reference'\n"
        "def get_camera_parames(cameras):\n    return calc_projected_points(None, None, None, None)\n")
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "lib" or k.startswith("lib.")}
    saved_path = list(sys.path)
    sys.path.insert(0, str(tmp_path / "ref"))
    sys.path.insert(0, ba_b200.PACKAGE_DIR)
    try:
        mod = importlib.import_module("lib.camera")
        assert mod.calc_projected_points is ba_b200.calc_projected_points
        assert mod.Camera.create((0, 0, -1), (0, 0, 1), f=1) == "reference camera"
        assert mod.get_camera_parames.__module__ == "lib._reference_camera"
        # the reference's own functions keep calling the reference's projection
        assert mod.get_camera_parames([]) == "reference"
    finally:
        sys.path[:] = saved_path
        for k in [k for k in sys.modules if k == "lib" or k.startswith("lib.")]:
            sys.modules.pop(k)
        sys.modules.update(saved)
