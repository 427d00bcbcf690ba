"""No result may depend on device memory the library did not write.  Needs a B200: `pytest -m gpu`.

Every engine buffer comes from the device's default memory pool (dev_alloc: cudaMallocAsync), the
pool keeps what engines free (retain_pool_memory), and the next engine of the process is built from
it -- the reference's class is used that way.  So a kernel that reads an element nobody wrote sees
whatever the previous user left: zeros so far, but NaN after a full-visibility list engine (its
bitmaps are 0xFFFFFFFF words).  Here the pool is filled with a 32-bit pattern before each scenario
runs, once with 0x00000000 and once with 0xFFFFFFFF (NaN doubles, int32 -1, full bitmaps), and every
output must be bitwise the same under both, and finite: sums run in a fixed order everywhere and
the only atomics are integer or bitwise, so any difference is a read of unwritten memory.

The reduced-system buffer `red` also lives across builds of one engine; the last tests fill it with
NaN before a build, and fill what its layout says is never read between the build and the solve.

The pool is driven through the CUDA driver API (ctypes on libcuda): stream-ordered allocation and
memset on the legacy stream, which dev_alloc uses too."""
import contextlib
import ctypes as C
import io

import numpy as np
import pytest

from oracle import ba_oracle as O
from test_gpu_parity import _check_random_scene

pytestmark = pytest.mark.gpu

ONES, ZEROS = 0xFFFFFFFF, 0x00000000
PATTERNS = (ZEROS, ONES)
C_DAMP = 1e-4


@pytest.fixture(scope="module")
def ba():
    import ba_b200

    return ba_b200


# ---- the device's default memory pool --------------------------------------------------------------
class _Pool:
    RELEASE_THRESHOLD, USED_MEM_CURRENT, USED_MEM_HIGH = 4, 7, 8  # CUmemPool_attribute

    def __init__(self):
        import torch

        torch.empty(1, device="cuda")  # the primary context, current on this thread
        self.drv = C.CDLL("libcuda.so.1")
        dev = C.c_int()
        self._check(self.drv.cuDeviceGet(C.byref(dev), torch.cuda.current_device()), "cuDeviceGet")
        self.pool = C.c_void_p()
        self._check(self.drv.cuDeviceGetDefaultMemPool(C.byref(self.pool), dev), "cuDeviceGetDefaultMemPool")
        # a freed block must stay in the pool (as create_engine also arranges) to be handed out again
        self.set(self.RELEASE_THRESHOLD, 2 ** 64 - 1)

    @staticmethod
    def _check(status, what):
        assert status == 0, f"{what} failed with CUresult {status}"

    def get(self, attr) -> int:
        v = C.c_uint64()
        self._check(self.drv.cuMemPoolGetAttribute(self.pool, attr, C.byref(v)), "cuMemPoolGetAttribute")
        return v.value

    def set(self, attr, value):
        v = C.c_uint64(value)
        self._check(self.drv.cuMemPoolSetAttribute(self.pool, attr, C.byref(v)), "cuMemPoolSetAttribute")

    def sync(self):
        self._check(self.drv.cuStreamSynchronize(None), "cuStreamSynchronize")

    def poison(self, word: int, nbytes: int):
        """Leave the pool holding nothing but `nbytes` of memory filled with the 32-bit `word`."""
        self.sync()
        self._check(self.drv.cuMemPoolTrimTo(self.pool, C.c_size_t(0)), "cuMemPoolTrimTo")
        nbytes = (nbytes + 3) // 4 * 4
        p = C.c_uint64()
        self._check(self.drv.cuMemAllocFromPoolAsync(C.byref(p), C.c_size_t(nbytes), self.pool, None),
                    "cuMemAllocFromPoolAsync")
        self._check(self.drv.cuMemsetD32Async(p, C.c_uint(word), C.c_size_t(nbytes // 4), None), "cuMemsetD32Async")
        self._check(self.drv.cuMemFreeAsync(p, None), "cuMemFreeAsync")
        self.sync()


@pytest.fixture(scope="module")
def pool(ba):
    return _Pool()


# The pattern the pool was last filled with (None: not poisoned); engines created while it is set
# check that they really received it.
_PATTERN = [None]

# buffers an engine has allocated but writes only from set_observations / linearize on
_UNWRITTEN_AT_CREATION = ("V", "GPT", "LINV", "Z", "U", "GCAM", "JP", "JC")


def _assert_holds_pattern(eng, names=_UNWRITTEN_AT_CREATION):
    word = _PATTERN[0]
    if word is None:
        return
    for name in names:
        got = eng.buffer(name).view(np.uint32)
        assert np.all(got == word), f"{name} did not come from the poisoned pool ({np.mean(got == word):.3f} of it did)"


def _new_engine(ba, n_points, n_cams, n_obs, f0, axis, dense):
    eng = ba.Engine(n_points, n_cams, n_obs, f0, axis, dense)
    _assert_holds_pattern(eng)
    return eng


def _mismatch(a, b, what):
    """None if a and b are equal bit for bit, else a description of where they differ."""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return f"{what}: {a.shape} {a.dtype} against {b.shape} {b.dtype}"
    if a.tobytes() == b.tobytes():
        return None
    rows = a.view(np.uint8).reshape(a.size, -1) != b.view(np.uint8).reshape(b.size, -1)
    diff = np.flatnonzero(rows.any(axis=1))
    return f"{what}: {diff.size} of {a.size} entries differ (first at flat index {diff[:5].tolist()})"


def _assert_all_equal(ref, got):
    bad = [m for name in ref if (m := _mismatch(np.asarray(ref[name]), np.asarray(got[name]), name))]
    assert not bad, "\n".join(bad)


def _run_poisoned(pool, scenario):
    """scenario() -> {name: array}; run on a clean pool to measure its footprint, then under each
    pattern; the outputs must be bitwise equal across the patterns and finite."""
    pool.sync()
    pool.set(_Pool.USED_MEM_HIGH, 0)
    base = pool.get(_Pool.USED_MEM_CURRENT)
    scenario()
    footprint = pool.get(_Pool.USED_MEM_HIGH) - base
    outs = {}
    for word in PATTERNS:
        pool.poison(word, int(footprint * 1.25) + (64 << 20))
        _PATTERN[0] = word
        try:
            outs[word] = scenario()
        finally:
            _PATTERN[0] = None
    ref, got = outs[ZEROS], outs[ONES]
    assert ref.keys() == got.keys()
    _assert_all_equal(ref, got)
    bad = [name for name, a in got.items() if np.asarray(a).dtype.kind == "f" and not np.all(np.isfinite(a))]
    assert not bad, f"not finite: {bad}"
    return ref


# ---- scenes ------------------------------------------------------------------------------------------
class _Scene:
    def __init__(self, sc, keep=None):
        n_per = np.diff(sc.obs_ptr)
        pt = np.repeat(np.arange(sc.n_points), n_per)
        cam = sc.obs_cam.astype(np.int64)
        xy = sc.obs_xy.reshape(-1, 2)
        if keep is not None:
            pt, cam, xy = pt[keep], cam[keep], xy[keep]
        ptr = np.concatenate(([0], np.cumsum(np.bincount(pt, minlength=sc.n_points)))).astype(np.int64)
        self.obs = O.ObsList(sc.n_points, sc.n_cams, pt, cam, np.ascontiguousarray(xy), ptr)
        self.X, self.R, self.t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, sc.axis)
        self.f, self.u = sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy()
        self.f0, self.axis = sc.f0, sc.axis
        self.full = bool(np.all(n_per == sc.n_cams)) and keep is None


def _random_scene(ba, n_cams, n_points, visibility, axis="x-up_z-forward", seed=None):
    sc = ba.scenes.make_scene(n_cams, n_points, seed=n_cams if seed is None else seed, visibility=visibility, axis=axis)
    return _Scene(sc)


def _zero_pair_scene(ba):
    """(40, 2000, 0.3) with cameras 0-9 and 30-39 sharing no point: of a point seen from both groups
    the smaller group's views are dropped (at least two views remain: make_scene gives three)."""
    sc = ba.scenes.make_scene(40, 2000, seed=40, visibility=0.3)
    cam = sc.obs_cam.astype(np.int64)
    pt = np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr))
    in_a, in_b = cam < 10, cam >= 30
    na, nb = np.bincount(pt, in_a, sc.n_points), np.bincount(pt, in_b, sc.n_points)
    drop_a = (na > 0) & (nb > 0) & (na <= nb)
    drop_b = (na > 0) & (nb > 0) & (na > nb)
    keep = ~((in_a & drop_a[pt]) | (in_b & drop_b[pt]))
    s = _Scene(sc, keep)
    vis = np.zeros((sc.n_points, sc.n_cams), dtype=bool)
    vis[s.obs.pt, s.obs.cam] = True
    assert vis.sum(axis=1).min() >= 2
    shared = vis[:, :10].astype(np.int64).T @ vis[:, 30:].astype(np.int64)
    assert not shared.any()
    # ... while every other pair shares points
    assert (vis.astype(np.int64).T @ vis.astype(np.int64)).astype(bool).sum() == 40 * 40 - 2 * 10 * 10
    return s


def _cam_chunks(n_sms, n_cams, n_obs):
    """create_engine's chunking of a camera's observations in camera_blocks_kernel / schur_diag_kernel."""
    chunks = max(1, (24 * n_sms + n_cams - 1) // n_cams)
    return min(chunks, max(1, (n_obs // n_cams + 1) // 1024))


def _empty_chunk_scene(ba):
    """(5, 9000, 0.7) with only 5 observations of camera 4 left and 25 200 in all (dropped from points
    that keep two or more views): 4 chunks per camera, and camera 4's 5 observations split 2, 2, 1
    and none."""
    import torch

    sc = ba.scenes.make_scene(5, 9000, seed=5, visibility=0.7)
    cam = sc.obs_cam.astype(np.int64)
    pt = np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr))
    views = np.bincount(pt, minlength=sc.n_points)
    keep = np.ones(cam.size, dtype=bool)
    kept4 = 0
    for o in np.flatnonzero(cam == 4):
        if kept4 < 5:
            kept4 += 1
        elif views[pt[o]] > 2:
            keep[o] = False
            views[pt[o]] -= 1
    # then the first view of points that keep three or more, down to 25 200 observations
    for o in np.flatnonzero(keep & (cam < 4)):
        if keep.sum() <= 25_200:
            break
        if views[pt[o]] > 3 and (o == 0 or pt[o - 1] != pt[o]):
            keep[o] = False
            views[pt[o]] -= 1
    s = _Scene(sc, keep)
    assert np.sum(s.obs.cam == 4) == 5
    n_sms = torch.cuda.get_device_properties(0).multi_processor_count
    chunks = _cam_chunks(n_sms, 5, s.obs.nobs)
    per = (5 + chunks - 1) // chunks
    assert chunks == 4 and per * (chunks - 1) >= 5, (chunks, per)
    return s


# ---- one engine through every phase -------------------------------------------------------------------
_PHASE_BUFFERS = ("JP", "JC", "V", "GPT", "U", "GCAM", "LINV", "Z", "DXI", "COST")


def _read_all(eng, phase, out):
    for name in _PHASE_BUFFERS + (("YT",) if eng.dense else ()):
        if phase == "linearize" and name in ("LINV", "Z"):
            continue  # K2b writes them, in build_reduced
        out[f"{phase}/{name}"] = eng.buffer(name)
    # of the reduced system only what its layout defines: the lower triangle of the n_rows block and
    # the 90 M tail (U_i and d_F staged by K3)
    red = eng.buffer("REDUCE")
    npad, nr = eng.n_pad, eng.rhs_row + 1
    out[f"{phase}/REDUCE"] = np.concatenate((red[: npad * npad].reshape(npad, npad)[:nr, :nr][np.tril_indices(nr)],
                                             red[npad * npad:]))


def _engine_scenario(ba, s, dense, lm_iters=3):
    def run():
        obs = s.obs
        eng = _new_engine(ba, obs.n_points, obs.n_cams, obs.nobs, s.f0, s.axis, dense)
        eng.set_observations(obs.ptr, None if dense else obs.cam.astype(np.int32), obs.xy)
        eng.set_state(s.X, s.R, s.t, s.f, s.u)
        out = {"E0": np.array([eng.cost(0)])}
        eng.linearize()
        _read_all(eng, "linearize", out)
        eng.build_reduced(C_DAMP)
        _read_all(eng, "build_reduced", out)
        eng.solve_trial(C_DAMP)
        _read_all(eng, "solve_trial", out)
        out["E_trial"] = np.array([eng.cost(1)])
        _read_all(eng, "cost", out)
        for name, a in zip("XRtfu", eng.get_state(1)):
            out[f"trial/{name}"] = a
        # a few iterations through the CUDA-graph loop, on the red / Lt / Winv the single phases left
        recs, st = eng.lm_run(2.0, 1e-8, lm_iters)
        out["records"] = np.array([(r.E_prev, r.E, r.delta, r.c, r.solves, r.count) for r in recs])
        out["lm_state"] = np.array([st.E, st.c, st.count, st.solves, st.status])
        for name, a in zip("XRtfu", eng.get_state(0)):
            out[f"final/{name}"] = a
        eng.close()
        return out
    return run


# (cameras, points, visibility, axis, dense): the regime each reaches, from test_gpu_parity.py and
# k4_cholesky.cu
ENGINE_SCENES = {
    "dense-30x1500": (30, 1500, 1.0, "x-up_z-forward", True),        # matrix-free, 64-tile DMMA SYRK, fused
                                                                     # Cholesky, one-CTA back substitution
    "dense-120x900": (120, 900, 1.0, "x-right_z-forward", True),    # 128-tile TMA SYRK, multi-panel fused Cholesky
    "dense-200x150-emu": (200, 150, 1.0, "x-up_z-forward", True),   # emulated SYRK with a ragged 256-tile row,
                                                                     # cluster back substitution
    "dense-400x700": (400, 700, 1.0, "x-up_z-forward", True),       # stored rows, two-level Cholesky, 128-tile updates
    "list-320x450": (320, 450, 0.3, "x-up_z-forward", False),       # pair lists, two-level Cholesky, grid back
                                                                     # substitution
    "list-70x3000-scan": (70, 3000, 0.9, "x-up_z-forward", False),  # bitmap-scan pair kernel
}
_ENV = {"dense-200x150-emu": {"BA_SYRK_EMU": "1"}, "list-70x3000-scan": {"BA_PAIRS_NO_LIST": "1"}}


def _scene_for(ba, key):
    if key == "list-zero-pairs":
        return _zero_pair_scene(ba), False
    if key == "list-empty-chunk":
        return _empty_chunk_scene(ba), False
    m, n, v, axis, dense = ENGINE_SCENES[key]
    return _random_scene(ba, m, n, v, axis), dense


@pytest.mark.parametrize("key", [*ENGINE_SCENES, "list-zero-pairs", "list-empty-chunk"])
def test_engine_outputs_do_not_depend_on_pool_contents(ba, pool, monkeypatch, key):
    for k, v in _ENV.get(key, {}).items():
        monkeypatch.setenv(k, v)
    s, dense = _scene_for(ba, key)
    _run_poisoned(pool, _engine_scenario(ba, s, dense))
    if "emu" in key:
        eng = ba.Engine(s.obs.n_points, s.obs.n_cams, s.obs.nobs, s.f0, s.axis, True)
        assert eng.syrk_emulated()
        eng.close()


def test_oracle_bar_holds_on_a_poisoned_pool(ba, pool):
    """The parity checks of one cheap scene (_check_one_linearisation) on a pool of NaNs."""
    pool.sync()
    pool.set(_Pool.USED_MEM_HIGH, 0)
    base = pool.get(_Pool.USED_MEM_CURRENT)
    _check_random_scene(ba, 30, 1500, 1.0, "x-up_z-forward")
    footprint = pool.get(_Pool.USED_MEM_HIGH) - base
    pool.poison(ONES, int(footprint * 1.25) + (64 << 20))
    _check_random_scene(ba, 30, 1500, 1.0, "x-up_z-forward")


# ---- covariances, the gauge on the device, the per-call entry points -------------------------------------
def _covariance_scenario(ba, s, dense):
    def run():
        obs = s.obs
        eng = _new_engine(ba, obs.n_points, obs.n_cams, obs.nobs, s.f0, s.axis, dense)
        eng.set_observations(obs.ptr, None if dense else obs.cam.astype(np.int32), obs.xy)
        eng.set_state(s.X, s.R, s.t, s.f, s.u)
        pc, cc, s2 = eng.covariance()
        eng.close()
        return {"point_cov": pc, "cam_cov": cc, "sigma2": np.array([s2])}
    return run


@pytest.mark.parametrize("m,n,vis,seed,dense", [(64, 400, 1.0, 64, True),
                                                (1000, 12000, 0.1, 3, False)])  # several batches (test_covariance.py)
def test_covariance_does_not_depend_on_pool_contents(ba, pool, m, n, vis, seed, dense):
    s = _random_scene(ba, m, n, vis, seed=seed)
    _run_poisoned(pool, _covariance_scenario(ba, s, dense))


def test_gauge_on_device_does_not_depend_on_pool_contents(ba, pool):
    """set_state_global / get_state_global (K6 and its scratch) through BundleAdjuster."""
    sc = ba.scenes.make_scene(12, 400, seed=5, visibility=0.6)

    def run():
        adj = ba.BundleAdjuster.from_observations(sc.obs_ptr, sc.obs_cam, sc.obs_xy, sc.X0, sc.K0, sc.R0, sc.t0,
                                                  f0=sc.f0, axis=sc.axis, gauge_on_device=True)
        _assert_holds_pattern(adj.engine)  # nothing linearised yet
        out = {f"normalised/{k}": a for k, a in zip("XRtfu", adj.engine.get_state(0))}
        with contextlib.redirect_stdout(io.StringIO()):
            X, K, R, t = adj.optimize(2.0, 1e-8, max_iter=4)
        out.update(X=X, K=K, R=R, t=t, E=np.array([[r["E_prev"], r["E"], r["c"]] for r in adj.records]))
        adj.engine.close()
        return out

    _run_poisoned(pool, run)


def test_per_call_paths_do_not_depend_on_pool_contents(ba, pool):
    """Projective depths (primary and dual), the rank-4 factorisation, the projection and one affine
    self-calibration: each allocates its scratch from the same pool."""
    import os

    sc = ba.scenes.make_scene(40, 3000, seed=3040, visibility=1.0)
    xd, _ = sc.dense_x()
    x = np.concatenate((xd / sc.f0, np.ones((sc.n_points, sc.n_cams, 1))), axis=2)
    rs = np.random.RandomState(7)
    W = rs.standard_normal((120, 4)) @ rs.standard_normal((4, 3000)) + 1e-3 * rs.standard_normal((120, 3000))
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "affine_calib.npz"))
    xl, f = [a.copy() for a in g["script_xy"]], g["script_f"]

    def run():
        out = {}
        out["primary/z"], out["primary/e"] = ba.projective_depth_primary(x, sc.f0, 1e-12, 4)
        out["dual/z"], out["dual/e"] = ba.projective_depth_dual(x, sc.f0, 1e-12, 4)
        out["rank4/M"], out["rank4/S"], out["rank4/s"] = ba.factorize_rank4(W)
        out["projection"] = np.stack(ba.calc_projected_points(sc.X0, sc.K0, sc.R0, sc.t0))
        out["affine/S"], out["affine/R"] = ba.paraperspective_self_calibration(xl, f)
        return {k: np.asarray(v, dtype=np.float64) for k, v in out.items()}

    _run_poisoned(pool, run)


# ---- the realistic sequence: a list engine's bitmaps become the next engine's buffers -----------------------
def test_dense_engine_after_a_full_visibility_list_engine(ba, pool):
    """A full-visibility list engine leaves 0xFFFFFFFF bitmap words (NaN doubles) in the pool; a dense
    engine of another shape built next must compute what it computes on a zeroed pool."""
    dense_scene = _random_scene(ba, 17, 333, 1.0)
    run_dense = _engine_scenario(ba, dense_scene, True)
    list_scene = _random_scene(ba, 30, 1500, 1.0)
    assert list_scene.full
    pool.poison(ZEROS, 1 << 30)
    ref = run_dense()
    pool.poison(ZEROS, 1 << 30)
    _engine_scenario(ba, list_scene, False)()
    _assert_all_equal(ref, run_dense())


# ---- the reduced-system buffer within one engine -----------------------------------------------------------
def _solve_outputs(eng):
    return {"DXI": eng.buffer("DXI"), "E_trial": np.array([eng.cost_values()[1]]),
            **{f"trial/{k}": a for k, a in zip("XRtfu", eng.get_state(1))}}


RED_SCENES = [("dense-30x1500", True), ("dense-30x1500", False), ("dense-120x900", True), ("dense-120x900", False),
              ("dense-200x150-emu", True), ("dense-400x700", True), ("dense-400x700", False),
              ("list-320x450", False), ("list-zero-pairs", False)]


@pytest.mark.parametrize("key,dense", RED_SCENES)
def test_reduced_system_reads_only_what_each_build_writes(ba, monkeypatch, key, dense):
    """1. red filled with NaN before build_reduced: the build and the solve give what they give on a
    fresh engine.  2. NaN written between build and solve into what the layout says is never read
    (the strict upper triangle of the n_rows block, every row and column from n_rows to n_pad): the
    solve is unchanged.  Compared bit for bit: DXI, the trial state and the trial cost."""
    import torch

    for k, v in _ENV.get(key, {}).items():
        monkeypatch.setenv(k, v)
    s, _ = _scene_for(ba, key)
    obs = s.obs
    eng = ba.Engine(obs.n_points, obs.n_cams, obs.nobs, s.f0, s.axis, dense)
    eng.set_observations(obs.ptr, None if dense else obs.cam.astype(np.int32), obs.xy)
    eng.set_state(s.X, s.R, s.t, s.f, s.u)
    eng.linearize()
    eng.build_reduced(C_DAMP)
    eng.solve_trial(C_DAMP)
    eng.cost(1)
    ref = _solve_outputs(eng)
    for name, a in ref.items():
        assert np.all(np.isfinite(a)), name

    red = eng.reduce_tensor()
    red.fill_(float("nan"))
    torch.cuda.synchronize()
    eng.build_reduced(C_DAMP)
    eng.solve_trial(C_DAMP)
    eng.cost(1)
    _assert_all_equal(ref, _solve_outputs(eng))  # NaN before the build

    npad, nr = eng.n_pad, eng.rhs_row + 1
    eng.build_reduced(C_DAMP)
    torch.cuda.synchronize()
    P = red[: npad * npad].view(npad, npad)
    P[:nr, :nr].masked_fill_(torch.ones(nr, nr, dtype=torch.bool, device=P.device).triu(1), float("nan"))
    P[nr:, :] = float("nan")
    P[:, nr:] = float("nan")
    torch.cuda.synchronize()
    eng.solve_trial(C_DAMP)
    eng.cost(1)
    _assert_all_equal(ref, _solve_outputs(eng))  # NaN outside the layout
    eng.close()
