"""Kernel instances that the camera count alone selects.  Needs a B200: `pytest -m gpu`.

Three choices depend on M only (kTabStride = 17 doubles per camera in shared memory):
  - dense engines re-derive the Jacobian rows (matrix-free, dense_matrix_free) while the camera
    table fits in 48 KB: M <= 361; above that K1 stores the rows as for a list engine;
  - K1 and the cost kernel stage the camera table in shared memory while it fits in 160 KB:
    M <= 1204; above that they read it from global memory;
  - the grid-wide back substitution runs min(n / 64, SMs) CTAs; from n = 9 M > 148 * 64 (M >= 1053
    on a B200) a CTA owns more than one 64-block.
The sweep checks the linearisation on both sides of the first two thresholds; the guard checks that
the large scenes of test_gpu_parity.py reach every instance."""
import re

import numpy as np
import pytest

from oracle import ba_oracle as O
from test_gpu_parity import CAMERA_COUNT_SCENES, _check_linearisation

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ba():
    import ba_b200

    return ba_b200


def _scene(ba, n_cams, n_points, visibility, axis="x-up_z-forward"):
    sc = ba.scenes.make_scene(n_cams, n_points, seed=n_cams, visibility=visibility, axis=axis)
    obs = O.ObsList(sc.n_points, sc.n_cams, np.repeat(np.arange(sc.n_points), np.diff(sc.obs_ptr)),
                    sc.obs_cam.astype(np.int64), sc.obs_xy, sc.obs_ptr)
    X, R, t = O.normalize_gauge(sc.X0, sc.R0, sc.t0, axis)
    return sc, obs, X, R, t, sc.K0[:, 0, 0].copy(), sc.K0[:, :2, 2].copy()


@pytest.mark.parametrize("dense", [True, False])
@pytest.mark.parametrize("n_cams", [360, 361, 362, 1204, 1205])
def test_linearisation_on_both_sides_of_the_camera_table_limits(ba, n_cams, dense):
    """cost(0), the Jacobian rows, V, d_P, U and d_F against the oracle at the last camera count
    below and the first above each limit, as a dense and as a list engine.  At 360 and 361 cameras the
    cost kernel's table (at most 48 KB) and its static scratch together need the opt-in to more than
    48 KB of shared memory; the launch failed there unless a larger engine had run first."""
    sc, obs, X, R, t, f, u = _scene(ba, n_cams, 40, 1.0)
    eng, _ = _check_linearisation(ba, obs, X, R, t, f, u, sc.f0, sc.axis, dense)
    assert eng.matrix_free() == (dense and n_cams <= 361)
    eng.close()


_INSTANCE = re.compile(r"\b(k1_residual_jacobian_kernel|cost_kernel|k2a_point_blocks_kernel|camera_blocks_kernel|"
                       r"k2b_point_solve_kernel|point_update_cost_kernel)\s*<([^<>]*)>")


def _instance(name):
    """(base name, (DENSE, second flag)) of a kernel name from the profiler, or None."""
    m = _INSTANCE.search(name)
    if not m:
        return None
    args = []
    for a in m.group(2).split(","):
        a = a.strip().replace("(bool)", "")
        args.append({"true": True, "1": True, "false": False, "0": False}.get(a, a))
    return m.group(1), tuple(args)


_TT, _TF, _FT, _FF = (True, True), (True, False), (False, True), (False, False)
EXPECTED = {
    "k1_residual_jacobian_kernel": {_TT, _TF, _FT, _FF},   # <DENSE, SMEM_TAB>
    "cost_kernel": {_TT, _TF, _FT, _FF},                   # <DENSE, SMEM_TAB>
    "k2a_point_blocks_kernel": {_TT, _TF, _FF},            # <DENSE, MF>
    "camera_blocks_kernel": {_TT, _TF, _FF},
    "k2b_point_solve_kernel": {_TT, _TF, _FF},
    "point_update_cost_kernel": {_TT, _TF, _FF},
}


def test_large_scenes_reach_every_instance(ba):
    """One linearisation, reduced system, trial step and cost of every scene of CAMERA_COUNT_SCENES
    (the dense ones also as list engines, as the bitwise dense / list comparison builds them) under
    the profiler: every template instance of K1, the cost kernel, K2a, the camera blocks, K2b and the
    point update runs, and one back substitution has more 64-blocks than the device has SMs."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    names = set()
    for n_cams, n_points, vis in CAMERA_COUNT_SCENES:
        sc, obs, X, R, t, f, u = _scene(ba, n_cams, n_points, vis)
        for dense in ([True, False] if sc.dense else [False]):
            eng = ba.Engine(obs.n_points, obs.n_cams, obs.nobs, sc.f0, sc.axis, dense)
            eng.set_observations(obs.ptr, None if dense else obs.cam.astype(np.int32), obs.xy)
            eng.set_state(X, R, t, f, u)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                eng.linearize()
                eng.build_reduced(1e-4)
                eng.solve_trial(1e-4)
                eng.cost(1)
                torch.cuda.synchronize()
            names |= {ev.key for ev in prof.key_averages()}
            eng.close()
    seen = {}
    for name in names:
        inst = _instance(name)
        if inst:
            seen.setdefault(inst[0], set()).add(inst[1])
    listing = "\n".join(sorted(names))
    for base, want in EXPECTED.items():
        missing = want - seen.get(base, set())
        assert not missing, f"{base}: instances {sorted(missing)} did not run; kernels seen:\n{listing}"
    nblk = max((9 * m + 63) // 64 for m, _, _ in CAMERA_COUNT_SCENES)
    assert nblk > sms, f"largest back substitution has {nblk} 64-blocks, the device {sms} SMs"
    assert any("chol_backsolve_grid_kernel" in n for n in names), listing
