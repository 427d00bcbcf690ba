"""ctypes binding of ``include/ba_b200.h`` (libba_b200.so).

Loading fails loudly: there is no CPU fallback behind this module.  Status codes map to the
exception types the reference raises (``ValueError`` for a bad axis,
``numpy.linalg.LinAlgError`` for a singular block -- reference
``lib/bundle_adjustment.py:28,128,146``) and ``RuntimeError`` otherwise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libba_b200.so")

(BA_OK, BA_ERR_INVALID, BA_ERR_CUDA, BA_ERR_SINGULAR, BA_ERR_STATE, BA_ERR_NO_DEVICE, BA_ERR_STALL,
 BA_ERR_COMM, BA_ERR_BARRIER) = range(9)
BA_COMM_HANDLE_BYTES = 88
BA_MEM_HOST, BA_MEM_DEVICE = 0, 1
BA_AXIS_X_RIGHT, BA_AXIS_X_UP = 0, 1
AXIS_CODES = {"x-right_z-forward": BA_AXIS_X_RIGHT, "x-up_z-forward": BA_AXIS_X_UP}

BUFFERS = {"JP": 0, "JC": 1, "V": 2, "GPT": 3, "U": 4, "GCAM": 5, "S": 6, "DXI": 7, "LINV": 8,
           "Z": 9, "REDUCE": 10, "COST": 11, "YT": 12}


class Problem(C.Structure):
    _fields_ = [("n_points", C.c_int64), ("n_obs", C.c_int64), ("n_cams", C.c_int32),
                ("axis", C.c_int32), ("f0", C.c_double), ("dense", C.c_int32), ("device", C.c_int32)]


class LMState(C.Structure):
    _fields_ = [("E", C.c_double), ("E_trial", C.c_double), ("c", C.c_double), ("delta", C.c_double),
                ("scale_factor", C.c_double), ("delta_tol", C.c_double), ("count", C.c_int32),
                ("max_iter", C.c_int32), ("solves", C.c_int32), ("iter_solves", C.c_int32),
                ("need_linearize", C.c_int32), ("accepted", C.c_int32), ("done", C.c_int32),
                ("status", C.c_int32), ("chol_fail", C.c_int32), ("max_retries", C.c_int32)]


class IterRecord(C.Structure):
    _fields_ = [("E_prev", C.c_double), ("E", C.c_double), ("delta", C.c_double), ("c", C.c_double),
                ("solves", C.c_int32), ("count", C.c_int32)]


# name -> (restype, argtypes); every entry must exist in the header and in the library
# (tests/test_cabi_symbols.py checks both directions).
_P = C.c_void_p
SIGNATURES = {
    "ba_version": (C.c_int, []),
    "ba_last_error": (C.c_char_p, []),
    "ba_device_count": (C.c_int, []),
    "ba_create": (C.c_int, [C.POINTER(Problem), C.POINTER(_P)]),
    "ba_destroy": (C.c_int, [_P]),
    "ba_set_observations": (C.c_int, [_P, _P, _P, _P, C.c_int, _P]),
    "ba_set_observations_dense": (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int, _P]),
    "ba_set_state": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "ba_get_state": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, C.c_int, _P]),
    "ba_set_state_global": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "ba_get_state_global": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.c_int, _P]),
    "ba_cost": (C.c_int, [_P, C.c_int, _P]),
    "ba_linearize": (C.c_int, [_P, _P]),
    "ba_build_reduced": (C.c_int, [_P, C.c_double, _P]),
    "ba_solve_trial": (C.c_int, [_P, C.c_double, _P]),
    "ba_lm_begin": (C.c_int, [_P, C.c_double, C.c_double, C.c_int, C.c_int, _P]),
    "ba_lm_phase_reduce": (C.c_int, [_P, _P]),
    "ba_lm_phase_solve": (C.c_int, [_P, _P]),
    "ba_lm_phase_decide": (C.c_int, [_P, _P]),
    "ba_lm_state_get": (C.c_int, [_P, C.POINTER(LMState), _P]),
    "ba_lm_state_post": (C.c_int, [_P, C.c_int, _P]),
    "ba_lm_state_wait": (C.c_int, [_P, C.c_int, C.POINTER(LMState)]),
    "ba_lm_iterate": (C.c_int, [_P, C.POINTER(LMState), _P]),
    "ba_lm_run": (C.c_int, [_P, C.c_double, C.c_double, C.c_int, C.c_int, C.POINTER(IterRecord),
                            C.c_int, C.POINTER(C.c_int), C.POINTER(LMState), _P]),
    "ba_lm_records": (C.c_int, [_P, C.POINTER(IterRecord), C.c_int, C.POINTER(C.c_int), _P]),
    "ba_reduce_buffer": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "ba_cost_buffer": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "ba_buffer_size": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int64)]),
    "ba_buffer_read": (C.c_int, [_P, C.c_int, _P, C.c_int64, _P]),
    "ba_reduced_layout": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "ba_comm_create": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "ba_comm_connect": (C.c_int, [_P, _P]),
    "ba_comm_disconnect": (C.c_int, [_P]),
    "ba_comm_world": (C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ba_launch_count": (C.c_int64, []),
    "ba_profile_enable": (C.c_int, [_P, C.c_int]),
    "ba_profile_get": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "ba_profile_reset": (C.c_int, [_P]),
    "ba_fp64_peak": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "ba_syrk_feed": (C.c_int, []),
    "ba_matrix_free": (C.c_int, [_P]),
    "ba_syrk_plan_info": (C.c_int, [C.c_int, C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                    C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "ba_syrk_emu_info": (C.c_int, [C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ba_syrk_emulated": (C.c_int, [_P]),
    "ba_projective_depth_primary": (C.c_int, [C.c_int, C.c_int64, C.c_int32, _P, C.c_double, C.c_double, C.c_int,
                                              _P, _P, C.POINTER(C.c_int), C.c_int, _P]),
    "ba_projective_depth_dual": (C.c_int, [C.c_int, C.c_int64, C.c_int32, _P, C.c_double, C.c_double, C.c_int,
                                           _P, _P, C.POINTER(C.c_int), C.c_int, _P]),
    "ba_depth_dual_probe": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "ba_factorize_rank4": (C.c_int, [C.c_int, C.c_int64, C.c_int32, _P, _P, _P, _P, C.c_int, _P]),
    "ba_factorize_centred_rank4": (C.c_int, [C.c_int, C.c_int64, C.c_int32, _P, _P, _P, _P, _P, C.c_int, _P]),
    "ba_project_points": (C.c_int, [C.c_int, C.c_int64, C.c_int32, _P, _P, _P, _P, _P, C.c_int, _P]),
}

_lib = None


def load() -> C.CDLL:
    """Load libba_b200.so (built in-tree by ``csrc/build.py`` / ``__graft_entry__.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python {os.path.join(PKG_DIR, 'csrc', 'build.py')}` "
            "(the engine has no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int) -> None:
    if status == BA_OK:
        return
    msg = load().ba_last_error().decode("utf-8", "replace")
    if status == BA_ERR_INVALID:
        raise ValueError(msg)
    if status == BA_ERR_SINGULAR:
        raise np.linalg.LinAlgError(msg)
    raise RuntimeError(f"ba_b200 error {status}: {msg}")
