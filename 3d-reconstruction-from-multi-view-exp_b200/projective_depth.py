"""Projective-depth iteration on the GPU: mirrors of the reference's
``_compute_projective_depth_primary_method`` (``lib/perspective_camera_calibration.py:61-144``) and
``_compute_projective_depth_dual_method`` (``:147-235``, the one ``euclidiean_reconstruction.py:42``
selects), the first stage of ``perspective_self_calibration``, and of ``factorization_method``
(``lib/factorization.py:5-15``), the stage after it -- the steps before bundle adjustment in the
perspective pipeline (SURVEY.md section 8f row 3).

Same arguments, return value and printed lines; the SVD and the per-point eigenproblems become a
Gram matrix on the FP64 tensor cores, one Jacobi eigen-solve and a per-point 4 x 4 problem behind
``ba_projective_depth_primary`` of the C ABI (``csrc/k7_projective_depth.cu``).  No CPU path.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _cabi
from .bundle_adjuster import _default_device


def _depth(symbol: str, x, f0: float, tolerance: float, max_iter: int, device: int | None):
    """``(z, errors)`` of the C entry point ``symbol`` (the primary or the dual method)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    if x.ndim != 3 or x.shape[2] != 3:
        raise ValueError("x must be (n_points, n_images, 3)")
    N, M = x.shape[:2]
    z = np.empty((N, M), dtype=np.float64)
    errors = np.empty(max(int(max_iter), 1), dtype=np.float64)  # the dual method runs one pass at least
    n_iter = C.c_int(0)
    fn = getattr(_cabi.load(), symbol)
    dev = _default_device() if device is None else int(device)
    _cabi.check(fn(dev, N, M, x.ctypes.data, float(f0), float(tolerance), int(max_iter), z.ctypes.data,
                   errors.ctypes.data, C.byref(n_iter), _cabi.BA_MEM_HOST, None))
    return z, errors[: n_iter.value].copy()


def projective_depth_primary(x, f0: float, tolerance: float, max_iter: int = 200, device: int | None = None):
    """``(z, errors)``: depths ``(n_points, n_images)`` and the reprojection error of every iteration."""
    return _depth("ba_projective_depth_primary", x, f0, tolerance, max_iter, device)


def compute_projective_depth_primary_method(x, f0: float, tolerance: float, max_iter: int = 200):
    """Reference signature and side effects (:61-63, :141, :144-145): prints one line per iteration."""
    z, errors = projective_depth_primary(x, f0, tolerance, max_iter)
    for count, E in enumerate(errors, start=1):
        print(f"Iteration {count}: reprojection_error = {E:.8}")
    if len(errors) >= max_iter:
        print("Did not converge because the maximum number of iterations was reached.")
    return z


MAX_IMAGES = 64  # the kernels keep one or two images per lane / a (3 M)^2 Gram matrix in one CTA's reach


def projective_depth_dual(x, f0: float, tolerance: float, max_iter: int = 50, device: int | None = None):
    """``(z, errors)`` of the dual method (:147-235) in O(n_images x n_points) memory."""
    return _depth("ba_projective_depth_dual", x, f0, tolerance, max_iter, device)


def compute_projective_depth_dual_method(x, f0: float, tolerance: float, max_iter: int = 50):
    """Reference signature and side effects (:147-150, :227-233): prints one line per pass."""
    z, errors = projective_depth_dual(x, f0, tolerance, max_iter)
    for count, E in enumerate(errors, start=1):
        print(f"Iteration {count}: reprojection_error = {E:.8}")
    if len(errors) >= max_iter:
        print("Did not converge because the maximum number of iterations was reached.")
    return z


def factorize_rank4(W, device: int | None = None):
    """``(M, S, sigma)``: rank-4 truncated SVD of ``W (n_rows, n_cols)``, ``n_rows <= 192``
    (``lib/factorization.py:5-15``): ``M (n_rows, 4)``, ``S (4, n_cols) = diag(sigma) V^T``."""
    W = np.asarray(W, dtype=np.float64)
    if W.ndim != 2:
        raise ValueError("W must be a matrix")
    n_rows, n_cols = W.shape
    Wt = np.ascontiguousarray(W.T)  # the reference passes `W.reshape(N, -1).T`: this is its base, no copy
    M = np.empty((n_rows, 4), dtype=np.float64)
    S = np.empty((4, n_cols), dtype=np.float64)
    sigma = np.empty(4, dtype=np.float64)
    lib = _cabi.load()
    dev = _default_device() if device is None else int(device)
    _cabi.check(lib.ba_factorize_rank4(dev, n_cols, n_rows, Wt.ctypes.data, M.ctypes.data, S.ctypes.data,
                                       sigma.ctypes.data, _cabi.BA_MEM_HOST, None))
    return M, S, sigma


def factorization_method(W, n_rank: int = 4):
    """Reference signature (``lib/factorization.py:5-7``): ``(M, S)``."""
    if n_rank != 4:
        raise ValueError("the GPU factorisation is the rank-4 one of the perspective pipeline")
    M, S, _ = factorize_rank4(W)
    return M, S
