"""The column maxima of the emulated dense Schur product are gathered by K2b as it writes Yt, and reset
before every K2b launch.  A maximum left over from an earlier build would give a column a smaller
exponent than its entries need now: builds at a large damping (Y shrinks) between builds at a small
one, and a covariance run (which runs K2b and K3 in a sequence of its own) before a build, must each
give P bit for bit as the exact host reconstruction from the Yt of that moment.  Needs a GPU."""
import numpy as np
import pytest

import ba_b200
from oracle import ba_oracle as O
from test_syrk_emulated_exact import _check_entries, _exact_P


def _assert_exact(eng, rng):
    npad = eng.n_pad
    P = eng.buffer("REDUCE")[: npad * npad].reshape(npad, npad).copy()
    Yt = eng.buffer("YT").reshape(-1, npad)
    moduli, bits = ba_b200.submodule("engine").syrk_emu_info(Yt.shape[0])
    idx = _check_entries(eng.rhs_row + 1, rng, n_random=5_000)
    want = _exact_P(Yt, list(moduli), bits, idx)
    got = P[idx[0], idx[1]]
    bad = np.flatnonzero(got.view(np.int64) != want.view(np.int64))
    assert bad.size == 0, f"{bad.size} of {got.size} entries differ from the exact reconstruction"
    return Yt


@pytest.mark.gpu
def test_column_maxima_follow_every_build(monkeypatch):
    monkeypatch.setenv("BA_SYRK_EMU", "1")
    axis = "x-up_z-forward"
    sc = ba_b200.scenes.make_scene(40, 900, seed=11, visibility=1.0, axis=axis)
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr)),
                    sc.obs_cam.astype(np.int64), sc.obs_xy, sc.obs_ptr)
    X, R, t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, axis)
    eng = ba_b200.Engine(obs.n_points, obs.n_cams, obs.nobs, sc.f0, axis, True)
    rng = np.random.default_rng(5)
    try:
        assert eng.syrk_emulated()
        eng.set_observations(obs.ptr, None, obs.xy)
        eng.set_state(X, R, t, sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy())
        eng.linearize()
        eng.build_reduced(1e-3)
        small = np.abs(_assert_exact(eng, rng)).max(axis=0)
        eng.build_reduced(1e6)
        large = np.abs(_assert_exact(eng, rng)).max(axis=0)
        assert np.all(large[small > 0] < small[small > 0] / 64), "the large damping should shrink every column"
        eng.build_reduced(1e-3)
        _assert_exact(eng, rng)
        eng.covariance()
        eng.build_reduced(1e6)
        _assert_exact(eng, rng)
    finally:
        eng.close()
