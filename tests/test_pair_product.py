"""The camera-pair half of the sparse Schur product (PairProduct, k3_schur_sparse.cu): its index is
rebuilt in place by every ba_set_observations, and ba_create refuses camera counts past the pair
kernels' launch limit.  Needs a B200: `pytest -m gpu`."""
import ctypes as C

import numpy as np
import pytest

from oracle import ba_oracle as O

pytestmark = pytest.mark.gpu

CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7  # cuda.h, CUmemPool_attribute


@pytest.fixture(scope="module")
def ba():
    import ba_b200

    return ba_b200


def _pool_bytes_in_use(device=0):
    """Bytes this process has allocated from the device's default memory pool, after a device
    synchronise (the engine's allocations and frees are stream-ordered on that pool)."""
    cu = C.CDLL("libcuda.so.1")
    assert cu.cuCtxSynchronize() == 0
    dev, pool, used = C.c_int(), C.c_void_p(), C.c_uint64()
    assert cu.cuDeviceGet(C.byref(dev), device) == 0
    assert cu.cuDeviceGetDefaultMemPool(C.byref(pool), dev) == 0
    assert cu.cuMemPoolGetAttribute(pool, CU_MEMPOOL_ATTR_USED_MEM_CURRENT, C.byref(used)) == 0
    return used.value


def test_setting_observations_again_replaces_the_pair_lists(ba):
    """Three ba_set_observations on one list engine with the same arrays: the pair lists of the first
    call (here ~400 MB) are replaced, not leaked, and the reduced system and an LM run (its solve
    graphs captured after the first call) come out bitwise the same."""
    sc = ba.scenes.make_scene(200, 20_000, seed=200, visibility=0.5)
    assert not sc.dense
    X, R, t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, sc.axis)
    f, u = sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy()
    cam = sc.obs_cam.astype(np.int32)
    eng = ba.Engine(sc.n_points, sc.n_cams, len(cam), sc.f0, sc.axis, dense=False)

    def reduced_and_run():
        eng.set_state(X, R, t, f, u)
        eng.cost(0)  # derives the camera table that the linearisation reads
        eng.linearize()
        eng.build_reduced(1e-3)
        red = eng.buffer("REDUCE")
        # what build_reduced writes: the lower triangle of P, its rhs row, U and d_F (the solve
        # factorises P in place, so the rest of the buffer holds what the last solve left there)
        npad, nfull = eng.n_pad, eng.n_full
        P = red[: npad * npad].reshape(npad, npad)
        red = np.concatenate([P[:nfull, :nfull][np.tril_indices(nfull)], P[eng.rhs_row, :nfull],
                              red[npad * npad:]])
        recs, _ = eng.lm_run(2.0, 1e-8, max_iter=3)
        return red, [(r.E_prev, r.E, r.c, r.solves) for r in recs]

    before = _pool_bytes_in_use()
    eng.set_observations(sc.obs_ptr, cam, sc.obs_xy)
    first = _pool_bytes_in_use()
    assert first - before >= 200 << 20  # the lists were built
    red0, run0 = reduced_and_run()
    for _ in range(2):
        eng.set_observations(sc.obs_ptr, cam, sc.obs_xy)
    assert _pool_bytes_in_use() <= first
    red2, run2 = reduced_and_run()
    eng.close()
    assert np.array_equal(red0.view(np.uint64), red2.view(np.uint64))
    assert run0 == run2


def test_create_refuses_cameras_past_the_camera_pair_limit(ba):
    """65 505 cameras make 2^31 pair items, more blocks than one launch takes: ba_create says so before
    it allocates anything (the reduced system alone would be 2.8 TB)."""
    with pytest.raises(ValueError, match="camera-pair limit"):
        ba.Engine(1, 65_505, 1, 1000.0, "x-up_z-forward", dense=False)
