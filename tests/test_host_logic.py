"""Host-side logic of the package (gauge, observation lists, scenes, sharding helpers) on CPU."""
import numpy as np
import pytest

import ba_b200
from conftest import SMALL_CASES, case_inputs, load_golden
from oracle import ba_oracle as O

gauge = ba_b200.submodule("gauge")
scenes = ba_b200.submodule("scenes")
sharded = ba_b200.submodule("sharded")
adjuster = ba_b200.submodule("bundle_adjuster")


@pytest.mark.parametrize("name", SMALL_CASES)
def test_gauge_normalisation_matches_reference(name):
    g = load_golden(name)
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    X, R, t = gauge.normalize(X0, R0, t0, axis)
    np.testing.assert_allclose(X, g["lin_nX"], rtol=0, atol=1e-14)
    np.testing.assert_allclose(R, g["lin_nR"], rtol=0, atol=1e-14)
    np.testing.assert_allclose(t, g["lin_nt"], rtol=0, atol=1e-14)
    np.testing.assert_allclose(R[0], np.eye(3), atol=1e-14)
    k = gauge.axis_component(axis)
    assert abs(abs(t[1, k]) - 1.0) < 1e-13
    # round trip (exact inverse only when the divisor was positive; the flip case is the
    # reference's documented quirk)
    L = gauge.baseline_length(R0, t0, axis)
    Xb, Rb, tb = gauge.denormalize(R0[0], t0[0], L, X, R, t)
    rel = t0[1] - t0[0]
    if np.sign(rel[k]) * (R0[0].T @ rel)[k] > 0:
        np.testing.assert_allclose(Xb, X0, atol=1e-12)
        np.testing.assert_allclose(tb, t0, atol=1e-12)
    np.testing.assert_allclose(Rb, R0, atol=1e-13)


def test_flip_case_has_negative_divisor():
    g = load_golden("small_flip_xup")
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    _, _, t = gauge.normalize(X0, R0, t0, axis)
    assert t[1, 1] == pytest.approx(-1.0, abs=1e-13)


def test_bad_axis_is_a_bare_value_error():
    with pytest.raises(ValueError):
        gauge.axis_component("z-up")
    with pytest.raises(ValueError):
        gauge.axis_component(None)


def test_make_K_layout():
    f = np.array([1.5, 2.0])
    u = np.array([[0.1, 0.2], [0.3, 0.4]])
    K = gauge.make_K(f, u, 0.7)
    np.testing.assert_array_equal(K, O.make_K(f, u, 0.7))
    assert K[0, 2, 2] == 0.7 and K[1, 1, 1] == 2.0 and K[1, 1, 2] == 0.4 and K[0, 1, 0] == 0.0


def test_observation_list_from_dense():
    g = load_golden("small_sparse_xup")
    x, vis, *_ = case_inputs(g)
    ol = adjuster.ObservationList.from_dense(x, vis)
    ref = O.ObsList.from_dense(x, vis)
    assert not ol.dense
    np.testing.assert_array_equal(ol.obs_ptr, ref.ptr)
    np.testing.assert_array_equal(ol.obs_cam, ref.cam)
    np.testing.assert_array_equal(ol.obs_xy, ref.xy)
    # dense: no camera array, non-contiguous input accepted (reference passes a transposed view)
    xt = np.ascontiguousarray(x.transpose(1, 0, 2)).transpose(1, 0, 2)
    assert not xt.flags.c_contiguous
    od = adjuster.ObservationList.from_dense(xt, None)
    assert od.dense and od.obs_cam is None and od.n_obs == x.shape[0] * x.shape[1]
    # a camera-major float64 block is handed over as it lies in memory (re-ordered on the device)
    assert od.obs_xy is None and od.dense_x is xt
    # anything else (another dtype, odd strides) is made contiguous on the host
    oc = adjuster.ObservationList.from_dense(xt.astype(np.float32), None)
    assert oc.dense_x is None
    np.testing.assert_array_equal(oc.obs_xy.reshape(x.shape), x.astype(np.float32).astype(np.float64))
    odd = np.zeros((x.shape[0], x.shape[1], 4))[:, :, :2]
    assert adjuster.ObservationList.from_dense(odd, None).dense_x is None
    # an all-true mask is the dense case
    assert adjuster.ObservationList.from_dense(x, np.ones(x.shape[:2], bool)).dense


def test_scene_generator_properties():
    sc = scenes.make_scene(12, 300, seed=5, visibility=0.25)
    counts = np.diff(sc.obs_ptr)
    assert counts.min() >= 3 and sc.obs_ptr[-1] == sc.nobs == sc.obs_cam.shape[0]
    pt = np.repeat(np.arange(sc.n_points), counts)
    for j in (0, 17, 299):  # cameras sorted within a point
        seg = sc.obs_cam[sc.obs_ptr[j]: sc.obs_ptr[j + 1]]
        assert np.all(np.diff(seg) > 0)
    # observations are projections of the ground truth + noise of the requested size
    f, u = sc.K_gt[:, 0, 0], sc.K_gt[:, :2, 2]
    exact = scenes.project_obs(sc.X_gt, f, u, sc.R_gt, sc.t_gt, sc.f0, pt, sc.obs_cam)
    resid = sc.obs_xy - exact
    assert 0.004 < resid.std() < 0.006
    # rotations are proper, cameras sit on the radius-5 hemisphere with x >= 0
    np.testing.assert_allclose(np.einsum("nij,nkj->nik", sc.R_gt, sc.R_gt), np.broadcast_to(np.eye(3), (12, 3, 3)), atol=1e-12)
    np.testing.assert_allclose(np.linalg.norm(sc.t_gt, axis=1), 5.0, atol=1e-12)
    assert np.all(sc.t_gt[:, 0] >= 0)
    x, vis = sc.dense_x()
    assert vis.sum() == sc.nobs and np.isfinite(x).all()
    # determinism
    sc2 = scenes.make_scene(12, 300, seed=5, visibility=0.25)
    np.testing.assert_array_equal(sc.obs_xy, sc2.obs_xy)


def test_scene_conventions_match_reference_camera_module():
    """look_at / projection against the reference's own lib/camera.py, through the cameras it made
    for tests/golden/projection.npz (oracle/gen_golden_projection.py): nine
    ``Camera.create(pos, target, f=1 + 0.1 i, f0=1)`` with the targets drawn from RandomState(7),
    then N(0, 0.01) noise added to K from the same stream."""
    g = load_golden("projection")
    rs = np.random.RandomState(7)
    tgt = np.array([rs.normal(0, 0.5, 3) for _ in range(9)])
    K = g["K"] - rs.normal(0, 0.01, g["K"].shape)
    f = 1.0 + 0.1 * np.arange(9)
    np.testing.assert_array_equal(K, gauge.make_K(f, np.zeros((9, 2)), 1.0))  # the stream is reproduced
    pos = g["t"]
    R = scenes.look_at(pos, tgt)
    np.testing.assert_allclose(R, g["R"], atol=1e-14)
    # the reference's projection of these cameras is pinned by the fixture through the oracle
    np.testing.assert_allclose(O.project_all(g["X"], g["K"], g["R"], pos), g["x"], rtol=1e-13, atol=1e-14)
    X = g["X"]
    proj = O.project_all(X, K, g["R"], pos)
    for i in range(9):
        mine = scenes.project_obs(X, f, np.zeros((9, 2)), R, pos, 1.0, np.arange(len(X)), np.full(len(X), i))
        np.testing.assert_allclose(mine, proj[i], atol=1e-13)
    # the reference's two known-answer projections (lib/camera.py:101-117)
    Xk = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=float)
    R1 = scenes.look_at(np.array([[0.0, 0, -1]]), np.array([[0.0, 0, 1]]))
    p1 = scenes.project_obs(Xk, np.ones(1), np.zeros((1, 2)), R1, np.array([[0.0, 0, -1]]), 1.0,
                            np.arange(4), np.zeros(4, int))
    np.testing.assert_allclose(p1, [[0, 0], [1, 0], [0, 1], [0, 0]], atol=1e-12)


def test_shard_bounds():
    b = sharded.shard_bounds(10, 3)
    assert b[0][0] == 0 and b[-1][1] == 10 and all(lo <= hi for lo, hi in b)
    assert [hi for _, hi in b[:-1]] == [lo for lo, _ in b[1:]]
    ptr = np.concatenate(([0], np.cumsum([1, 1, 1, 1, 20, 1, 1, 1, 1, 1])))
    b2 = sharded.shard_bounds(10, 2, ptr)
    assert b2[0][0] == 0 and b2[-1][1] == 10
    loads = [ptr[hi] - ptr[lo] for lo, hi in b2]
    assert max(loads) <= 25  # the heavy point does not drag everything onto one rank


def test_oracle_sharded_partials_sum_to_the_whole():
    """The quantities a sharded run all-reduces are additive over point shards."""
    g = load_golden("small_sparse_xup")
    x, vis, X0, K0, R0, t0, axis, f0 = case_inputs(g)
    obs = O.ObsList.from_dense(x, vis)
    X, R, t = O.normalize_gauge(X0, R0, t0, axis)
    f, u = K0[:, 0, 0].copy(), K0[:, :2, 2].copy()
    lin = O.linearize(obs, X, f, u, R, t, f0)
    A, b, _ = O.reduced_system(obs, lin, 1e-3)
    M = obs.n_cams
    Psum = np.zeros_like(A)
    bsum = np.zeros_like(b)
    Usum = np.zeros((M, 9, 9))
    for lo, hi in sharded.shard_bounds(obs.n_points, 3, obs.ptr):
        sub = obs.subset_points(lo, hi)
        ls = O.linearize(sub, X[lo:hi], f, u, R, t, f0)
        As, bs, _ = O.reduced_system(sub, ls, 0.0)  # c = 0 keeps U undamped in As
        Ublk = np.zeros_like(A)
        for i in range(M):
            Ublk[9 * i: 9 * i + 9, 9 * i: 9 * i + 9] = ls.U[i]
        Usum += ls.U
        # recompute with the damped point blocks only (the U damping is applied after the sum)
        As2, bs2, _ = O.reduced_system(sub, ls, 1e-3)
        Ud = np.zeros_like(A)
        for i in range(M):
            blk = ls.U[i].copy()
            blk[np.arange(9), np.arange(9)] *= 1 + 1e-3
            Ud[9 * i: 9 * i + 9, 9 * i: 9 * i + 9] = blk
        Psum += Ud - As2  # = sum_j F^T E^-1 F of the shard
        bsum += bs2
    Utot = np.zeros_like(A)
    for i in range(M):
        blk = Usum[i].copy()
        blk[np.arange(9), np.arange(9)] *= 1 + 1e-3
        Utot[9 * i: 9 * i + 9, 9 * i: 9 * i + 9] = blk
    np.testing.assert_allclose(Utot - Psum, A, rtol=0, atol=1e-10 * np.abs(A).max())
    np.testing.assert_allclose(bsum, b, rtol=0, atol=1e-10 * np.abs(b).max())


@pytest.mark.parametrize("n_cams,n_points,tile", [(50, 10_000, 64), (50, 10_000, 128), (200, 100_000, 128),
                                                  (17, 333, 64), (120, 900, 128), (2, 5, 64),
                                                  (200, 12_500, 128), (114, 4_000, 128), (320, 450, 128),
                                                  (57, 10_000, 128), (228, 20_000, 128)])
def test_schur_product_plan_covers_every_tile_once(n_cams, n_points, tile):
    """The host-side scheduler of the dense Schur product (K3): the work items must cut every
    lower-triangle tile's K range into consecutive pieces without gaps or overlaps, and the
    modelled schedule of the benchmark shapes must stay within 15 % of the perfectly balanced one
    (library self-check through the C ABI; no device involved).  128-tile plans have folded diagonal
    tiles and -- when at most 16 rows are left over (200 cameras: n_pad = 14 x 128 + 16; 57 and 228
    cameras: 8 rows) -- the ragged last tile row folded into "tall" tiles of the row above, whose
    thin tiles then own no items but one second partial-tile slot per piece of the tall tile."""
    import ctypes as C

    import ba_b200

    cabi = ba_b200.submodule("_cabi")
    lib = cabi.load()
    ni, nt, mk, ideal = C.c_int(), C.c_int(), C.c_double(), C.c_double()
    cabi.check(lib.ba_syrk_plan_info(n_cams, n_points, tile, 148, C.byref(ni), C.byref(nt), C.byref(mk),
                                     C.byref(ideal)))
    n_pad = (9 * n_cams + 1 + 7) // 8 * 8
    nt1 = (n_pad + tile - 1) // tile
    assert nt.value == nt1 * (nt1 + 1) // 2
    assert ni.value >= nt.value
    if n_points >= 10_000:
        assert ideal.value / mk.value > 0.85
