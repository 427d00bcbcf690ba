"""CPU oracle of the marginal covariances (``ba_covariance`` / ``BundleAdjuster.covariance``).

Everything at the given state, undamped, gauge unknowns removed, in the normalised frame and the
camera parameter order (f, u0, v0, t, w) of ``ba_oracle.linearize``.  H = [[U, W], [W^T, V]] is
the Gauss-Newton Hessian with the reference's factor 2 (H = 2 J^T J), so the covariance
sigma^2 (J^T J)^-1 is 2 sigma^2 H^-1 with sigma^2 = E / (2 n_obs - (3N + 9M - 7)).

Two independent routes:
  * ``covariance_full``  -- the definition: assemble H, delete the gauge rows and columns, invert
    (small scenes only);
  * ``covariance_schur`` -- the reduced camera system S = L L^T: camera blocks of S^-1 from L^-1,
    point blocks V^-1 + V^-1 W_j^T S^-1 W_j V^-1 for a chosen subset of points.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

from . import ba_oracle as O


def sigma2(E: float, n_obs: int, n_points: int, n_cams: int) -> float:
    dof = 2 * n_obs - (3 * n_points + 9 * n_cams - 7)
    if dof <= 0:
        raise ValueError(f"covariance needs more residuals than unknowns (2 n_obs = {2 * n_obs}, "
                         f"unknowns = {3 * n_points + 9 * n_cams - 7})")
    return E / dof


def _full_hessian(obs: O.ObsList, lin: O.Linearization) -> np.ndarray:
    N, M = obs.n_points, obs.n_cams
    nc = 9 * M
    H = np.zeros((nc + 3 * N, nc + 3 * N))
    for i in range(M):
        H[9 * i: 9 * i + 9, 9 * i: 9 * i + 9] = lin.U[i]
    for j in range(N):
        H[nc + 3 * j: nc + 3 * j + 3, nc + 3 * j: nc + 3 * j + 3] = lin.V[j]
    for o in range(obs.nobs):
        j, i = int(obs.pt[o]), int(obs.cam[o])
        H[nc + 3 * j: nc + 3 * j + 3, 9 * i: 9 * i + 9] = lin.W[o]
        H[9 * i: 9 * i + 9, nc + 3 * j: nc + 3 * j + 3] = lin.W[o].T
    return H


def covariance_full(obs: O.ObsList, X, f, u, R, t, f0, axis):
    """(cov_X (N, 3, 3), cov_cam (M, 9, 9), sigma2) by inverting the full gauge-reduced Hessian."""
    N, M = obs.n_points, obs.n_cams
    lin = O.linearize(obs, X, f, u, R, t, f0)
    s2 = sigma2(lin.cost, obs.nobs, N, M)
    removed, _ = O.gauge_indices(M, axis)
    keep = np.ones(9 * M + 3 * N, dtype=bool)
    keep[removed] = False
    H = _full_hessian(obs, lin)
    Hinv = np.zeros_like(H)
    Hinv[np.ix_(keep, keep)] = np.linalg.inv(H[np.ix_(keep, keep)])
    C = 2.0 * s2 * Hinv
    cam = np.stack([C[9 * i: 9 * i + 9, 9 * i: 9 * i + 9] for i in range(M)])
    nc = 9 * M
    pts = np.stack([C[nc + 3 * j: nc + 3 * j + 3, nc + 3 * j: nc + 3 * j + 3] for j in range(N)])
    return pts, cam, s2


def covariance_schur(obs: O.ObsList, X, f, u, R, t, f0, axis, points=None, schur: str = "dense"):
    """(cov_X (len(points), 3, 3), cov_cam (M, 9, 9), sigma2) through the reduced camera system.

    ``points`` selects the point blocks (default: all); ``schur="sparse"`` assembles S with the
    sparsity-aware C kernel of ``ba_oracle.reduced_system_sparse`` (1000-camera scenes)."""
    N, M = obs.n_points, obs.n_cams
    lin = O.linearize(obs, X, f, u, R, t, f0)
    s2 = sigma2(lin.cost, obs.nobs, N, M)
    _, kept = O.gauge_indices(M, axis)
    if schur == "sparse":
        A, _, Vinv = O.reduced_system_sparse(obs, lin, 0.0)
    else:
        A, _, Vinv = O.reduced_system(obs, lin, 0.0)
    L = np.linalg.cholesky(A[np.ix_(kept, kept)])
    Linv, info = sla.lapack.dtrtri(L, lower=1)
    if info != 0:
        raise np.linalg.LinAlgError("singular reduced system")
    # S^-1 = L^-T L^-1: its diagonal blocks are Gram matrices of columns of L^-1
    Linv_full = np.zeros((len(kept), 9 * M))
    Linv_full[:, kept] = Linv
    cam = np.stack([Linv_full[:, 9 * i: 9 * i + 9].T @ Linv_full[:, 9 * i: 9 * i + 9] for i in range(M)])
    sel = np.arange(N) if points is None else np.asarray(points)
    pts = np.empty((len(sel), 3, 3))
    pos = {int(c): k for k, c in enumerate(kept)}
    for k, j in enumerate(sel):
        a, b = int(obs.ptr[j]), int(obs.ptr[j + 1])
        Wj = np.zeros((len(kept), 3))  # camera x point block of H, gauge rows deleted
        for o in range(a, b):
            i = int(obs.cam[o])
            for p in range(9):
                if 9 * i + p in pos:
                    Wj[pos[9 * i + p]] = lin.W[o][:, p]
        Z = Linv @ (Wj @ Vinv[j])  # L^-1 W_j V_j^-1
        pts[k] = Vinv[j] + Z.T @ Z
    return 2.0 * s2 * pts, 2.0 * s2 * cam, s2
