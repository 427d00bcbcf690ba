"""Host-side mirror of the reference ``BundleAdjuster`` (``lib/bundle_adjustment.py:10-206``).

Same constructor, ``optimize`` and ``get_log`` signatures, array conventions, printed lines
and exception types; the Levenberg-Marquardt loop itself runs on the GPU behind the C ABI.
Additions that the reference does not have (all keyword-only / separate constructors):
  * ``BundleAdjuster.from_observations`` -- observation-list (CSR by point) ingestion, so the
    1000 x 1M sparse configurations never build the dense ``(N, M, 2)`` array;
  * ``process_group`` -- points sharded over ranks (one engine per GPU); per inner solve the
    partial reduced system and the trial cost are summed over the ranks, by default
    (``exchange="peer"`` whenever the group runs on NCCL, i.e. one GPU per rank) by the
    library's own kernels over NVLink peer memory, otherwise (``exchange="collective"``) by
    two ``torch.distributed`` all-reduces;
  * ``max_retries`` -- a cap on inner solves per iteration (the reference loops forever, :118);
  * ``gauge_on_device`` -- the O(N) gauge normalisation / de-normalisation passes (:208-258) run
    as CUDA kernels (``ba_set_state_global`` / ``ba_get_state_global``) instead of NumPy.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import gauge
from .engine import Engine


@dataclass
class ObservationList:
    """Visible (point, camera) pairs sorted by point, then camera (CSR by point)."""

    obs_ptr: np.ndarray  # (N+1,) int64
    obs_cam: np.ndarray | None  # (nobs,) int32; None when dense
    obs_xy: np.ndarray | None  # (nobs, 2) float64; None when `dense_x` carries the block
    n_cams: int
    dense: bool
    # the caller's dense ``x (N, M, 2)`` itself when it is one point-major or camera-major block of
    # float64: uploaded as it lies in memory and re-ordered on the device (ba_set_observations_dense)
    dense_x: np.ndarray | None = None

    @property
    def n_points(self) -> int:
        return int(self.obs_ptr.shape[0] - 1)

    @property
    def n_obs(self) -> int:
        if self.obs_xy is None:
            return int(self.dense_x.shape[0] * self.dense_x.shape[1])
        return int(self.obs_xy.shape[0])

    @staticmethod
    def from_dense(x, visibility_index=None) -> "ObservationList":
        """Reference layout: ``x (N, M, 2)`` (any strides) and an optional bool mask (N, M)."""
        N, M = x.shape[:2]
        if visibility_index is None or bool(np.all(visibility_index)):
            ptr = np.arange(N + 1, dtype=np.int64) * M
            if isinstance(x, np.ndarray) and x.dtype == np.float64 and x.ndim == 3 and x.shape[2] == 2 \
                    and x.strides[2] == 8 and (x.strides[0], x.strides[1]) in ((16 * M, 16), (16, 16 * N)):
                # what both reference scripts pass: np.stack(x_list).transpose(1, 0, 2)
                return ObservationList(ptr, None, None, M, True, dense_x=x)
            xy = np.ascontiguousarray(x, dtype=np.float64).reshape(N * M, 2)
            return ObservationList(ptr, None, xy, M, True)
        vis = np.asarray(visibility_index, dtype=bool)
        pt, cam = np.nonzero(vis)
        xy = np.ascontiguousarray(np.asarray(x, dtype=np.float64)[pt, cam])
        ptr = np.concatenate(([0], np.cumsum(vis.sum(axis=1)))).astype(np.int64)
        return ObservationList(ptr, cam.astype(np.int32), xy, M, False)


class BundleAdjuster:
    def __init__(self, x, init_X, init_K, init_R, init_t, f0=1.0, visibility_index=None,
                 axis="x-right_z-forward", *, observations: ObservationList | None = None,
                 device: int | None = None, process_group=None, max_retries: int = 200,
                 exchange: str = "auto", gauge_on_device: bool = False):
        gauge.axis_component(axis)  # ValueError() for an unknown axis (:28)
        init_X = np.asarray(init_X, dtype=np.float64)
        init_R = np.asarray(init_R, dtype=np.float64)
        init_t = np.asarray(init_t, dtype=np.float64)
        init_K = np.asarray(init_K)  # may be a read-only broadcast view; never written (:45-48)

        # saved to return to the caller's frame (:23-33)
        self._R0 = init_R[0].copy()
        self._t0 = init_t[0].copy()
        self._c0c1_len = gauge.baseline_length(init_R, init_t, axis)
        self._axis = axis
        self._f0 = float(f0)
        self._x = x  # kept by reference like the reference does (:37)

        obs = observations if observations is not None else ObservationList.from_dense(x, visibility_index)
        self._obs = obs
        self._n_points = init_X.shape[0]
        self._n_images = init_R.shape[0]
        if obs.n_points != self._n_points or obs.n_cams != self._n_images:
            raise ValueError("observations do not match init_X / init_R")

        # normalised frame (:40-42); intrinsics (:45-48) as fresh arrays
        self._gauge_on_device = bool(gauge_on_device)
        if self._gauge_on_device:
            self._X = self._R = self._t = None  # the normalised state exists on the device only
        else:
            self._X, self._R, self._t = gauge.normalize(init_X, init_R, init_t, axis)
        self._f = np.array(init_K[:, 0, 0], dtype=np.float64)
        self._u = np.array(init_K[:, :2, 2], dtype=np.float64)

        self._group = process_group
        self._max_retries = int(max_retries)
        self._log: list[dict] = []
        self.records: list[dict] = []  # per accepted iteration: E_prev, E, delta, c, solves

        if device is None:
            device = _default_device()
        self._engine = Engine(self._n_points, self._n_images, obs.n_obs, self._f0, axis, obs.dense, device)
        if obs.dense_x is not None:
            self._engine.set_observations_dense(obs.dense_x)
        else:
            self._engine.set_observations(obs.obs_ptr, obs.obs_cam, obs.obs_xy)
        if self._gauge_on_device:
            self._engine.set_state_global(init_X, init_R, init_t, self._f, self._u)
        else:
            self._engine.set_state(self._X, self._R, self._t, self._f, self._u)
        self._peer_exchange = False
        self._quiet = False  # sharded runs: only rank 0 prints the iteration lines (:188)
        if exchange not in ("auto", "peer", "collective"):
            raise ValueError("exchange must be 'auto', 'peer' or 'collective'")
        if process_group is not None and exchange != "collective":
            import torch.distributed as dist

            world = dist.get_world_size(process_group)
            if exchange == "peer" or (str(dist.get_backend(process_group)) == "nccl" and 2 <= world <= 8):
                if world >= 2:
                    self._engine.comm_attach(dist, process_group)
                    self._peer_exchange = True
                    self._quiet = dist.get_rank(process_group) != 0

    @classmethod
    def from_observations(cls, obs_ptr, obs_cam, obs_xy, init_X, init_K, init_R, init_t, f0=1.0,
                          axis="x-right_z-forward", dense=False, **kw):
        n_cams = np.asarray(init_R).shape[0]
        obs = ObservationList(np.asarray(obs_ptr, dtype=np.int64),
                              None if dense else np.asarray(obs_cam, dtype=np.int32),
                              np.asarray(obs_xy, dtype=np.float64).reshape(-1, 2), n_cams, bool(dense))
        return cls(None, init_X, init_K, init_R, init_t, f0=f0, axis=axis, observations=obs, **kw)

    @property
    def engine(self) -> Engine:
        return self._engine

    # ------------------------------------------------------------------------------------------
    def optimize(self, scale_factor=10.0, delta_tol=1e-8, max_iter=100, is_debug=False):
        """Minimise the reprojection error over X, K, R, t (reference :77-202)."""
        eng = self._engine
        self.records = []
        if self._group is not None and not self._peer_exchange:
            from .sharded import run_sharded

            run_sharded(self, scale_factor, delta_tol, max_iter, is_debug)
        elif is_debug:
            eng.lm_begin(scale_factor, delta_tol, max_iter, self._max_retries)
            self._log.clear()
            self._log_state(float(eng.cost_values()[0]))  # entry 0 = initial state (:89-98)
            while True:
                st = eng.lm_iterate()
                self._after_accept(st, is_debug=True)
                if st.done:
                    break
        else:
            recs, st = eng.lm_run(scale_factor, delta_tol, max_iter, self._max_retries)
            for r in recs:
                self._record(r.E_prev, r.E, r.delta, r.c, r.solves, r.count)

        if self._gauge_on_device:
            return eng.get_state_global(0)  # (:198-202) on the device
        self._X, self._R, self._t, self._f, self._u = eng.get_state(0)
        # back to the caller's frame (:198-200)
        self._X, self._R, self._t = gauge.denormalize(self._R0, self._t0, self._c0c1_len,
                                                      self._X, self._R, self._t)
        return self._X, gauge.make_K(self._f, self._u, self._f0), self._R, self._t

    def covariance(self):
        """Marginal covariances at the current state (after ``optimize``: the solution), in the
        caller's frame that ``optimize`` returns: ``(cov_X (N, 3, 3), cov_cam (M, 9, 9), sigma2)``,
        cameras in the order (f, u0, v0, t, w).  sigma2 = E / (2 n_obs - n_unknowns) scales
        (J^T J)^-1; the 7 gauge-pinned camera parameters have zero rows and columns.  Raises
        ``numpy.linalg.LinAlgError`` for a point seen fewer than twice or an indefinite system."""
        if self._group is not None:
            raise RuntimeError("covariance of a sharded adjuster is not supported")
        cov_X, cov_cam, sigma2 = self._engine.covariance()
        cov_X, cov_cam = gauge.covariance_to_caller(self._R0, self._c0c1_len, cov_X, cov_cam)
        return cov_X, cov_cam, sigma2

    def get_log(self):
        """Per-iteration points / camera log in the normalised frame (:204-206)."""
        return self._log

    # ------------------------------------------------------------------------------------------
    def _record(self, E_prev, E, delta, c, solves, count):
        self.records.append({"E_prev": E_prev, "E": E, "delta": delta, "c": c, "solves": solves,
                             "count": count})
        if not self._quiet:
            print(f"Iteration {count}: reprojection_error_delta = {np.float64(delta)}")  # :188

    def _log_state(self, E):
        X, R, t, _, _ = self._engine.get_state(0)
        self._log.append({"points": X, "basis": R, "pos": t, "reprojection_error": np.float64(E)})

    def _after_accept(self, st, is_debug):
        if st.count > len(self.records):
            recs = self._engine.lm_records()
            for r in recs[len(self.records):]:
                self._record(r.E_prev, r.E, r.delta, r.c, r.solves, r.count)
                if is_debug:
                    self._log_state(r.E)


def _default_device() -> int:
    """torch's current device if the caller already uses torch with CUDA up, else device 0 (torch
    is never imported from here, see ``engine._current_stream``)."""
    import sys

    torch = sys.modules.get("torch")
    try:
        if torch is not None and torch.cuda.is_available() and torch.cuda.is_initialized():
            return int(torch.cuda.current_device())
    except Exception:  # pragma: no cover
        pass
    return 0
