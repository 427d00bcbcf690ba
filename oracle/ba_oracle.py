"""CPU oracle for the perspective-camera LM bundle adjustment hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is part of the product: only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl
reference`` legs may import it, and only as the checker / the timed CPU baseline.  The
product path (the CUDA engine behind ``include/ba_b200.h``) never routes through here.

What this is: a float64 NumPy *observation-list* restatement of the algorithm of
``/root/reference/lib/bundle_adjustment.py`` (class ``BundleAdjuster``).  The reference
works on dense ``(n_points, n_images, ...)`` arrays and materialises an ``(N, n, n)``
temporary (``lib/bundle_adjustment.py:135``), so it cannot hold anything beyond ~50 cameras
x 10k points.  This restatement evaluates exactly the same quantities per *visible*
observation and reduces them per point / per camera, so it also runs the large configs.

Parity pin: the reference has no tests or golden vectors for this path (SURVEY.md section 4),
so the oracle is pinned against *outputs of the reference itself*, produced in the build
container by ``oracle/gen_golden.py`` (imports ``/root/reference`` unmodified) and committed
under ``tests/golden/``; ``tests/test_oracle_golden.py`` replays them.

Line map (all ``lib/bundle_adjustment.py`` unless noted):
  projection ............ :283-307          -> ``camera_tables`` / ``project``
  derivative table ...... :309-427          -> ``linearize``
  gradients ............. :429-517          -> ``Linearization.g_pt`` / ``g_cam``
  GN blocks ............. :519-664          -> ``Linearization.V`` / ``W`` / ``U``
  damping, Schur, solve . :118-152          -> ``solve_damped``
  update ................ :260-281, lib/utils.py:10-29 -> ``apply_update`` / ``rodrigues``
  cost .................. :666-677          -> ``cost``
  LM control ............ :100-195          -> ``OracleBundleAdjuster.optimize``
  gauge ................. :62-72, :208-258  -> ``gauge_indices`` / ``normalize_gauge`` /
                                               ``denormalize_gauge``
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

AXES = ("x-right_z-forward", "x-up_z-forward")


# --------------------------------------------------------------------------------------
# observation list
# --------------------------------------------------------------------------------------
@dataclass
class ObsList:
    """Visible (point, camera) pairs, sorted by point then camera (CSR by point)."""

    n_points: int
    n_cams: int
    pt: np.ndarray  # (nobs,) int64 point index of each observation
    cam: np.ndarray  # (nobs,) int64 camera index of each observation
    xy: np.ndarray  # (nobs, 2) float64 measured image coordinates
    ptr: np.ndarray  # (n_points + 1,) int64 CSR offsets

    @property
    def nobs(self) -> int:
        return int(self.pt.shape[0])

    @staticmethod
    def from_dense(x: np.ndarray, vis: np.ndarray | None = None) -> "ObsList":
        """Dense ``x (N, M, 2)`` + bool mask ``(N, M)`` (reference layout, :36-37, :56-60)."""
        n_points, n_cams = x.shape[:2]
        if vis is None:
            vis = np.ones((n_points, n_cams), dtype=bool)
        vis = np.asarray(vis, dtype=bool)
        pt, cam = np.nonzero(vis)  # row-major order == sorted by point, then camera
        xy = np.ascontiguousarray(np.asarray(x, dtype=np.float64)[pt, cam])
        counts = np.bincount(pt, minlength=n_points)
        ptr = np.concatenate(([0], np.cumsum(counts))).astype(np.int64)
        return ObsList(n_points, n_cams, pt.astype(np.int64), cam.astype(np.int64), xy, ptr)

    def subset_points(self, lo: int, hi: int) -> "ObsList":
        """Observations of points ``lo:hi`` re-indexed from 0 (used for point shards)."""
        a, b = int(self.ptr[lo]), int(self.ptr[hi])
        return ObsList(
            hi - lo,
            self.n_cams,
            self.pt[a:b] - lo,
            self.cam[a:b],
            self.xy[a:b],
            self.ptr[lo : hi + 1] - self.ptr[lo],
        )


# --------------------------------------------------------------------------------------
# gauge (reference :23-33, :62-72, :208-258)
# --------------------------------------------------------------------------------------
def gauge_axis_index(axis: str) -> int:
    """Component of the camera-0 frame whose baseline is pinned (0: x-right, 1: x-up)."""
    if axis == "x-right_z-forward":
        return 0
    if axis == "x-up_z-forward":
        return 1
    raise ValueError()


def gauge_indices(n_cams: int, axis: str) -> tuple[np.ndarray, np.ndarray]:
    """(removed, kept) indices into the full 9M camera-parameter vector (:62-72)."""
    k = gauge_axis_index(axis)
    removed = np.array([3, 4, 5, 6, 7, 8, 9 + 3 + k])
    keep = np.ones(9 * n_cams, dtype=bool)
    keep[removed] = False
    return removed, np.nonzero(keep)[0]


def normalize_gauge(X, R, t, axis):
    """Camera 0 -> identity/origin, baseline component k -> +-1 (:208-240).

    The divisor ``s`` takes its *sign* from the world-frame component of ``t1 - t0`` and
    its *magnitude* from the camera-0-frame component -- a quirk of the reference that is
    kept verbatim (SURVEY.md section 8 a2).
    """
    k = gauge_axis_index(axis)
    R0 = R[0]
    dX = X - t[0]
    dt = t - t[0]
    s = np.sign(dt[1, k]) * (R0.T @ dt[1])[k]
    return (dX @ R0) / s, R0.T @ R, (dt @ R0) / s


def baseline_length(R, t, axis):
    """``c0c1_len`` saved by the constructor (:23-26)."""
    k = gauge_axis_index(axis)
    return np.abs(R[0][:, k] @ (t[1] - t[0]))


def denormalize_gauge(R0, t0, scale, X, R, t):
    """Back to the caller's frame (:242-258)."""
    return (scale * X) @ R0.T + t0, R0 @ R, (scale * t) @ R0.T + t0


# --------------------------------------------------------------------------------------
# projection, cost, linearisation
# --------------------------------------------------------------------------------------
def camera_tables(f, u, R, t, f0):
    """Rows of ``P[:, :, :3] = K R^T`` (:283-302): gradients of (p, q, r) w.r.t. X."""
    gp = f[:, None] * R[:, :, 0] + u[:, :1] * R[:, :, 2]
    gq = f[:, None] * R[:, :, 1] + u[:, 1:] * R[:, :, 2]
    gr = f0 * R[:, :, 2]
    return gp, gq, gr


def project(obs: ObsList, X, f, u, R, t, f0):
    """(p, q, r) per visible observation (:299-305), plus the pieces reused later."""
    gp, gq, gr = camera_tables(f, u, R, t, f0)
    d = X[obs.pt] - t[obs.cam]
    gpo, gqo, gro = gp[obs.cam], gq[obs.cam], gr[obs.cam]
    p = np.einsum("ok,ok->o", gpo, d)
    q = np.einsum("ok,ok->o", gqo, d)
    r = np.einsum("ok,ok->o", gro, d)
    return p, q, r, d, gpo, gqo, gro


def cost(obs: ObsList, X, f, u, R, t, f0) -> float:
    """E = sum over visible observations of squared reprojection error (:666-677)."""
    p, q, r, *_ = project(obs, X, f, u, R, t, f0)
    e0 = p / r - obs.xy[:, 0] / f0
    e1 = q / r - obs.xy[:, 1] / f0
    return float(np.sum(e0 * e0 + e1 * e1))


@dataclass
class Linearization:
    e: np.ndarray  # (nobs, 2)   residuals
    Jx: np.ndarray  # (nobs, 2, 3) d e / d X_j           = (a_X, b_X) / r^2
    Jc: np.ndarray  # (nobs, 2, 9) d e / d (f,u0,v0,t,w) = (a_c, b_c) / r^2
    cost: float
    g_pt: np.ndarray  # (N, 3)    d_P  (:429-469)
    g_cam: np.ndarray  # (M, 9)   d_F before the gauge entries are dropped (:471-509)
    V: np.ndarray  # (N, 3, 3)    matE (:519-556)
    U: np.ndarray  # (M, 9, 9)    diagonal blocks of matG (:618-653)
    W: np.ndarray  # (nobs, 3, 9) block of matF for (point, camera) of the observation (:558-605)


def _segment_sum(index: np.ndarray, values: np.ndarray, size: int) -> np.ndarray:
    """sum of ``values[o]`` over observations with ``index[o] == k`` for k < size."""
    flat = values.reshape(values.shape[0], -1)
    out = np.empty((size, flat.shape[1]))
    for c in range(flat.shape[1]):
        out[:, c] = np.bincount(index, weights=flat[:, c], minlength=size)
    return out.reshape((size,) + values.shape[1:])


def linearize(obs: ObsList, X, f, u, R, t, f0) -> Linearization:
    p, q, r, d, gp, gq, gr = project(obs, X, f, u, R, t, f0)
    fo, uo = f[obs.cam], u[obs.cam]

    # a_theta = r dp/dtheta - p dr/dtheta, b_theta likewise (:450, :459, :492, :501)
    aX = r[:, None] * gp - p[:, None] * gr
    bX = r[:, None] * gq - q[:, None] * gr

    ac = np.empty((obs.nobs, 9))
    bc = np.empty((obs.nobs, 9))
    # focal length (:336-338): dp/df = (p - u0/f0 r)/f, dr/df = 0
    ac[:, 0] = r * ((p - uo[:, 0] / f0 * r) / fo)
    bc[:, 0] = r * ((q - uo[:, 1] / f0 * r) / fo)
    # principal point (:350-356): dp/du0 = r/f0, dq/dv0 = r/f0
    ac[:, 1] = r * (r / f0)
    ac[:, 2] = 0.0
    bc[:, 1] = 0.0
    bc[:, 2] = r * (r / f0)
    # translation (:368-376): d/dt = -d/dX
    ac[:, 3:6] = -aX
    bc[:, 3:6] = -bX
    # rotation (:391-396): d(p,q,r)/dw = grad x (X - t)
    cp, cq, cr = np.cross(gp, d), np.cross(gq, d), np.cross(gr, d)
    ac[:, 6:9] = r[:, None] * cp - p[:, None] * cr
    bc[:, 6:9] = r[:, None] * cq - q[:, None] * cr

    r2 = (r * r)[:, None]
    Jx = np.stack((aX / r2, bX / r2), axis=1)
    Jc = np.stack((ac / r2, bc / r2), axis=1)
    e = np.stack((p / r - obs.xy[:, 0] / f0, q / r - obs.xy[:, 1] / f0), axis=1)

    # gradient = 2 sum J^T e, Gauss-Newton blocks = 2 sum J^T J  (:462-467, :546-554, ...)
    g_pt = 2.0 * _segment_sum(obs.pt, np.einsum("ok,oka->oa", e, Jx), obs.n_points)
    g_cam = 2.0 * _segment_sum(obs.cam, np.einsum("ok,oka->oa", e, Jc), obs.n_cams)
    V = 2.0 * _segment_sum(obs.pt, np.einsum("oka,okb->oab", Jx, Jx), obs.n_points)
    U = 2.0 * _segment_sum(obs.cam, np.einsum("oka,okb->oab", Jc, Jc), obs.n_cams)
    W = 2.0 * np.einsum("oka,okb->oab", Jx, Jc)
    return Linearization(e, Jx, Jc, float(np.sum(e * e)), g_pt, g_cam, V, U, W)


# --------------------------------------------------------------------------------------
# damped Schur solve (:118-152)
# --------------------------------------------------------------------------------------
def damp_point_blocks(V, c):
    Vc = V.copy()
    i = np.arange(3)
    Vc[:, i, i] *= 1.0 + c
    return Vc


def reduced_system(obs: ObsList, lin: Linearization, c: float, chunk_points: int = 4096):
    """Full (9M x 9M) ``G_c - sum_j F_j^T E_j^-1 F_j`` and rhs before gauge deletion.

    Returns (A_full, b_full, Vinv).  Point chunks are expanded to the reference's dense
    ``matF`` rows ``(3, 9M)`` (:608) so the contraction is one BLAS GEMM per chunk instead of
    the reference's ``(N, n, n)`` temporary (:135).
    """
    M, N = obs.n_cams, obs.n_points
    nfull = 9 * M
    Vinv = np.linalg.inv(damp_point_blocks(lin.V, c))  # (:128)

    A = np.zeros((nfull, nfull))
    for i in range(M):  # block_diag of U_i with the diagonal scaled by 1+c (:123-125, :656)
        blk = lin.U[i].copy()
        k = np.arange(9)
        blk[k, k] *= 1.0 + c
        A[9 * i : 9 * i + 9, 9 * i : 9 * i + 9] = blk
    b = -lin.g_cam.reshape(-1).copy()

    cols = 9 * obs.cam[:, None] + np.arange(9)[None, :]  # (nobs, 9)
    for lo in range(0, N, chunk_points):
        hi = min(N, lo + chunk_points)
        a, z = int(obs.ptr[lo]), int(obs.ptr[hi])
        if a == z:
            continue
        F = np.zeros((hi - lo, 3, nfull))
        rows = (obs.pt[a:z] - lo)[:, None, None]
        F[rows, np.arange(3)[None, :, None], cols[a:z, None, :]] = lin.W[a:z]
        EF = Vinv[lo:hi] @ F  # (cn, 3, 9M)
        F2 = F.reshape(-1, nfull)
        A -= F2.T @ EF.reshape(-1, nfull)  # (:132-135)
        b += np.einsum("jkn,jk->n", EF, lin.g_pt[lo:hi])  # (:138-143), E^-1 symmetric
    return A, b, Vinv


def reduced_system_sparse(obs: ObsList, lin: Linearization, c: float):
    """The same (A_full, b_full, Vinv) as ``reduced_system`` without multiplying the zero blocks
    of cameras that do not see a point: per point only the (9 m_j) x (9 m_j) sub-matrix of its
    own cameras is updated (``oracle/ba_schur_sparse.c``, plain C + OpenMP).  This is the CPU
    formulation the 1000-camera configurations are timed on -- sum_j 3 (9 m_j)(9 m_j + 1) flops
    instead of the dense 2 * 3 * n^2 * N (SURVEY.md section 8d)."""
    from . import build_c

    lib = build_c.load()
    M = obs.n_cams
    nfull = 9 * M
    Vinv = np.ascontiguousarray(np.linalg.inv(damp_point_blocks(lin.V, c)))  # (:128)
    A = np.zeros((nfull, nfull))
    k = np.arange(9)
    for i in range(M):  # block_diag of U_i with the diagonal scaled by 1+c (:123-125, :656)
        blk = lin.U[i].copy()
        blk[k, k] *= 1.0 + c
        A[9 * i: 9 * i + 9, 9 * i: 9 * i + 9] = blk
    b = -lin.g_cam.reshape(-1).copy()
    W = np.ascontiguousarray(lin.W)
    g_pt = np.ascontiguousarray(lin.g_pt)
    ptr = np.ascontiguousarray(obs.ptr, dtype=np.int64)
    cam = np.ascontiguousarray(obs.cam, dtype=np.int64)
    lib.ba_oracle_schur_sparse(obs.n_points, M, ptr.ctypes.data, cam.ctypes.data, W.ctypes.data,
                               Vinv.ctypes.data, g_pt.ctypes.data, A.ctypes.data, b.ctypes.data)
    return A, b, Vinv


def schur_flops_sparse(obs: ObsList) -> float:
    """sum_j 3 (9 m_j)(9 m_j + 1): multiply-adds x 2 of the lower triangle of the Schur product."""
    m = np.diff(obs.ptr).astype(np.float64)
    return float(np.sum(3.0 * (9.0 * m) * (9.0 * m + 1.0)))


def solve_damped(obs: ObsList, lin: Linearization, c: float, axis: str, chunk_points: int = 4096,
                 schur: str = "dense", solver: str = "lu", reduced=None):
    """One inner LM solve: returns (delta_xi_full (M,9), delta_X (N,3), A_red, b_red).

    ``schur="sparse"`` uses the sparsity-aware C restatement; ``solver="cholesky"`` replaces the
    reference's LU (:146) by LAPACK ``dposv`` -- half the flops at n = 8993, and SURVEY.md section 6
    measured the effect on the cost trajectory at <= 3e-14 relative (A is SPD).  ``reduced``: the
    (A_full, b_full, Vinv) of this ``lin`` and ``c`` when the caller has formed it already."""
    _, kept = gauge_indices(obs.n_cams, axis)
    if reduced is not None:
        A, b, Vinv = reduced
    elif schur == "sparse":
        A, b, Vinv = reduced_system_sparse(obs, lin, c)
    else:
        A, b, Vinv = reduced_system(obs, lin, c, chunk_points)
    A_red = A[np.ix_(kept, kept)]
    b_red = b[kept]
    if solver == "cholesky":
        import scipy.linalg as sla

        dxi_red = sla.solve(A_red, b_red, assume_a="pos", check_finite=False)
    else:
        dxi_red = np.linalg.solve(A_red, b_red)  # (:146) LU, as in the reference
    dxi = np.zeros(9 * obs.n_cams)
    dxi[kept] = dxi_red  # re-insert zeros for the pinned entries (:267)
    dxi = dxi.reshape(obs.n_cams, 9)
    # back-substitution (:152): dX_j = -E_j^-1 (F_j dxi + d_P_j)
    Fdxi = _segment_sum(obs.pt, np.einsum("oab,ob->oa", lin.W, dxi[obs.cam]), obs.n_points)
    dX = -np.einsum("jab,jb->ja", Vinv, Fdxi + lin.g_pt)
    return dxi, dX, A_red, b_red


# --------------------------------------------------------------------------------------
# parameter update (:260-281, lib/utils.py:10-29)
# --------------------------------------------------------------------------------------
def rodrigues(w: np.ndarray) -> np.ndarray:
    """Axis-angle -> rotation; exact identity iff w == 0 exactly (lib/utils.py:14-15)."""
    if not np.any(w):
        return np.eye(3)
    th = np.sqrt(w @ w)
    l = w / th
    c, s = np.cos(th), np.sin(th)
    skew = np.array([[0.0, -l[2], l[1]], [l[2], 0.0, -l[0]], [-l[1], l[0], 0.0]])
    return (1.0 - c) * np.outer(l, l) + c * np.eye(3) + s * skew


def apply_update(X, f, u, R, t, dxi, dX):
    dR = np.stack([rodrigues(w) for w in dxi[:, 6:9]])
    return X + dX, f + dxi[:, 0], u + dxi[:, 1:3], dR @ R, t + dxi[:, 3:6]


def make_K(f, u, f0):
    """(:283-289)"""
    K = np.zeros((f.shape[0], 3, 3))
    K[:, 0, 0] = f
    K[:, 1, 1] = f
    K[:, :2, 2] = u
    K[:, 2, 2] = f0
    return K


# --------------------------------------------------------------------------------------
# LM driver with the reference's class API
# --------------------------------------------------------------------------------------
class OracleBundleAdjuster:
    """Same constructor / ``optimize`` / ``get_log`` contract as the reference class (:10-206)."""

    def __init__(self, x, init_X, init_K, init_R, init_t, f0=1.0, visibility_index=None,
                 axis="x-right_z-forward", obs: ObsList | None = None):
        gauge_axis_index(axis)  # ValueError for unknown axis (:28)
        self._axis = axis
        self._R0 = np.array(init_R[0], dtype=np.float64)
        self._t0 = np.array(init_t[0], dtype=np.float64)
        self._scale = baseline_length(init_R, init_t, axis)
        self._obs = obs if obs is not None else ObsList.from_dense(x, visibility_index)
        self._X, self._R, self._t = normalize_gauge(
            np.asarray(init_X, dtype=np.float64), np.asarray(init_R, dtype=np.float64),
            np.asarray(init_t, dtype=np.float64), axis)
        self._f = np.array(init_K[:, 0, 0], dtype=np.float64)
        self._u = np.array(init_K[:, :2, 2], dtype=np.float64)
        self._f0 = float(f0)
        self._log: list[dict] = []
        self.trace: list[dict] = []  # per accepted iteration: E, c used, number of inner solves

    def optimize(self, scale_factor=10.0, delta_tol=1e-8, max_iter=100, is_debug=False,
                 verbose=True, chunk_points=4096, schur="dense", solver="lu"):
        obs, f0 = self._obs, self._f0
        E = cost(obs, self._X, self._f, self._u, self._R, self._t, f0)
        if is_debug:
            self._log.clear()
            self._log.append({"points": self._X.copy(), "basis": self._R.copy(),
                              "pos": self._t.copy(), "reprojection_error": E})
        self.trace = [{"E": E, "c": None, "solves": 0}]
        c = 0.0001
        count = 0
        while True:
            lin = linearize(obs, self._X, self._f, self._u, self._R, self._t, f0)
            solves = 0
            while True:
                dxi, dX, _, _ = solve_damped(obs, lin, c, self._axis, chunk_points, schur, solver)
                solves += 1
                tX, tf, tu, tR, tt = apply_update(self._X, self._f, self._u, self._R, self._t, dxi, dX)
                E_ = cost(obs, tX, tf, tu, tR, tt, f0)
                if E_ > E:
                    c *= scale_factor
                else:
                    break
            self._X, self._f, self._u, self._R, self._t = tX, tf, tu, tR, tt
            if is_debug:
                self._log.append({"points": self._X.copy(), "basis": self._R.copy(),
                                  "pos": self._t.copy(), "reprojection_error": E_})
            self.trace.append({"E": E_, "c": c, "solves": solves})
            count += 1
            delta = np.abs(E_ - E)
            if verbose:
                print(f"Iteration {count}: reprojection_error_delta = {delta}")
            if delta <= delta_tol or count >= max_iter:
                break
            E = E_
            c /= scale_factor
        self._X, self._R, self._t = denormalize_gauge(self._R0, self._t0, self._scale,
                                                      self._X, self._R, self._t)
        return self._X, make_K(self._f, self._u, f0), self._R, self._t

    def get_log(self):
        return self._log


# ---- batched re-projection (reference lib/camera.py:13, :28-32, :74-81) -----------------------
def project_all(X, K, R, t):
    """``calc_projected_points`` for all cameras at once: ``(M, N, 2)``.

    Per camera P = K [R^T | -R^T t] (``get_camera_matrix``, :13), X_ext @ P^T, then the
    perspective division by the third component (``_perspective_projection``, :28-32)."""
    X = np.asarray(X, dtype=np.float64)
    K = np.asarray(K, dtype=np.float64)
    R = np.asarray(R, dtype=np.float64)
    t = np.asarray(t, dtype=np.float64)
    Rt = np.transpose(R, (0, 2, 1))
    E = np.concatenate([Rt, -(Rt @ t[:, :, None])], axis=2)  # (M, 3, 4)
    P = K @ E
    X_ext = np.hstack([X, np.ones((X.shape[0], 1))])
    proj = np.einsum("nc,mrc->mnr", X_ext, P)
    return proj[:, :, :2] / proj[:, :, 2:3]
