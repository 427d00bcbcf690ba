"""Host-side gauge handling of the reference constructor / epilogue (O(N + M) NumPy).

Mirrors reference ``lib/bundle_adjustment.py``: the saved camera-0 frame and baseline length
(:23-33), ``_transform_to_normalize_coodinates`` (:208-240) and
``_inverse_transform_to_global_coordinates`` (:242-258).  This is the host form, used by the
reference-signature constructor; ``gauge_on_device=True`` runs the same transforms as CUDA
kernels behind ``ba_set_state_global`` / ``ba_get_state_global`` (``csrc/k6_gauge.cu``).
"""
from __future__ import annotations

import numpy as np

AXIS_COMPONENT = {"x-right_z-forward": 0, "x-up_z-forward": 1}


def axis_component(axis: str) -> int:
    try:
        return AXIS_COMPONENT[axis]
    except (KeyError, TypeError):
        raise ValueError() from None  # the reference raises a bare ValueError (:28, :232)


def baseline_length(R, t, axis: str):
    """|R0[:, k] . (t1 - t0)| (:24, :26)."""
    k = axis_component(axis)
    return np.abs(R[0][:, k] @ (t[1] - t[0]))


def normalize(X, R, t, axis: str):
    """Scene expressed in camera 0's frame with the pinned baseline component scaled to +-1.

    Quirk kept from the reference (:228-234): the divisor takes its sign from the *world*
    component k of t1 - t0 but its magnitude from the camera-0-frame component, so it can be
    negative (point-reflected scene); ``denormalize`` multiplies by the positive length.
    """
    k = axis_component(axis)
    R0 = R[0]
    rel_t = t - t[0]
    s = np.sign(rel_t[1, k]) * (R0.T @ rel_t[1])[k]
    return ((X - t[0]) @ R0) / s, R0.T @ R, (rel_t @ R0) / s


def denormalize(R0, t0, length, X, R, t):
    """(:254-256)"""
    return (length * X) @ R0.T + t0, R0 @ R, (length * t) @ R0.T + t0


def make_K(f, u, f0):
    """K = [[f,0,u0],[0,f,v0],[0,0,f0]] per camera (:283-289)."""
    K = np.zeros((f.shape[0], 3, 3))
    K[:, 0, 0] = f
    K[:, 1, 1] = f
    K[:, 0, 2] = u[:, 0]
    K[:, 1, 2] = u[:, 1]
    K[:, 2, 2] = f0
    return K


def covariance_jacobians(R0, length):
    """Jacobians of ``denormalize`` at the solution: points ``length R0``, cameras
    T = blockdiag(I_3, length R0, R0) over (f, u0, v0, t, w).  The rotation update is
    R <- exp([w]x) R, so R0 exp([w]x) R = exp([R0 w]x) R0 R maps w by R0.  The sign of the
    divisor (``normalize``) cancels in T S T^T."""
    Jx = length * np.asarray(R0)
    T = np.zeros((9, 9))
    T[:3, :3] = np.eye(3)
    T[3:6, 3:6] = Jx
    T[6:, 6:] = R0
    return Jx, T


def covariance_to_caller(R0, length, cov_X, cov_cam):
    """Normalised-frame covariances -> the caller's frame: Jx S Jx^T per point, T S T^T per camera."""
    Jx, T = covariance_jacobians(R0, length)
    out_X = None if cov_X is None else Jx @ cov_X @ Jx.T
    return out_X, T @ cov_cam @ T.T
