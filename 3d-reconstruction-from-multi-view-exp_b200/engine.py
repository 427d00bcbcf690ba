"""Thin Python handle over the C-ABI engine (``include/ba_b200.h``).

Host code passes NumPy arrays (host pointers) or CUDA tensors (raw device pointers); PyTorch is
used only to hand device memory across (``data_ptr()``, the current stream, and tensor views of
the two buffers a sharded run all-reduces).
"""
from __future__ import annotations

import atexit
import ctypes as C
import sys
import weakref

import numpy as np

from . import _cabi

# Engines still alive when the interpreter exits are destroyed from an atexit hook, i.e. while the
# CUDA runtime is still up: an engine that is only collected during interpreter finalisation (the
# reference scripts keep theirs in a module global) would call into a torn-down CUDA context from
# __del__ -- a segmentation fault at exit.
_live_engines: "weakref.WeakSet[Engine]" = weakref.WeakSet()


@atexit.register
def _close_live_engines():
    for eng in list(_live_engines):
        try:
            eng.close()
        except Exception:
            pass


def _current_stream(device: int) -> int:
    """torch's current CUDA stream on `device` if the CALLER already uses torch with CUDA up, else
    the default stream.  torch is never imported from here: a caller that has not imported it (the
    reference scripts) cannot have a torch stream current, the import costs seconds, and an import
    that fails half-way (e.g. under a stub `matplotlib` whose modules answer every attribute) leaves
    extension modules behind that crash the interpreter at exit."""
    torch = sys.modules.get("torch")
    try:
        if torch is not None and torch.cuda.is_available() and torch.cuda.is_initialized():
            return int(torch.cuda.current_stream(device).cuda_stream)
    except Exception:  # pragma: no cover - a broken torch: default stream
        pass
    return 0


def _ptr(a, dtype):
    """(pointer, mem, keepalive) of a NumPy array or a CUDA tensor; None -> (None, HOST, None)."""
    if a is None:
        return None, _cabi.BA_MEM_HOST, None
    if hasattr(a, "data_ptr") and getattr(a, "is_cuda", False):
        import torch

        want = {np.float64: torch.float64, np.int64: torch.int64, np.int32: torch.int32}[dtype]
        if a.dtype != want or not a.is_contiguous():
            raise ValueError("device tensors must be contiguous and of the expected dtype")
        return a.data_ptr(), _cabi.BA_MEM_DEVICE, a
    arr = np.ascontiguousarray(a, dtype=dtype)
    return arr.ctypes.data, _cabi.BA_MEM_HOST, arr


class _DeviceView:
    """Exposes a raw device range through ``__cuda_array_interface__`` (for torch.as_tensor)."""

    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False),
                                         "version": 2, "strides": None}


class Engine:
    def __init__(self, n_points: int, n_cams: int, n_obs: int, f0: float, axis: str, dense: bool,
                 device: int = 0):
        if axis not in _cabi.AXIS_CODES:
            raise ValueError()
        self._lib = _cabi.load()
        self.n_points, self.n_cams, self.n_obs = int(n_points), int(n_cams), int(n_obs)
        self.dense, self.device, self.f0, self.axis = bool(dense), int(device), float(f0), axis
        prob = _cabi.Problem(self.n_points, self.n_obs, self.n_cams, _cabi.AXIS_CODES[axis], self.f0,
                             1 if dense else 0, self.device)
        h = C.c_void_p()
        _cabi.check(self._lib.ba_create(C.byref(prob), C.byref(h)))
        self._h = h
        npad, nfull, rhs = C.c_int32(), C.c_int32(), C.c_int32()
        _cabi.check(self._lib.ba_reduced_layout(self._h, C.byref(npad), C.byref(nfull), C.byref(rhs)))
        self.n_pad, self.n_full, self.rhs_row = npad.value, nfull.value, rhs.value
        _live_engines.add(self)

    # -- life cycle ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._comm = None  # exchange windows outlive engines (recycled, never freed)
            self._lib.ba_destroy(self._h)
            self._h = None

    def __del__(self):
        if sys is None or sys.is_finalizing():  # too late to talk to CUDA; the atexit hook ran already
            return
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self) -> int:
        return _current_stream(self.device)

    # -- data ---------------------------------------------------------------------------------
    def set_observations(self, obs_ptr, obs_cam, obs_xy):
        p_ptr, m1, k1 = _ptr(obs_ptr, np.int64)
        p_cam, m2, k2 = _ptr(None if self.dense else obs_cam, np.int32)
        p_xy, m3, k3 = _ptr(obs_xy, np.float64)
        mems = {m for p, m in ((p_ptr, m1), (p_cam, m2), (p_xy, m3)) if p is not None}
        if len(mems) != 1:
            raise ValueError("observation arrays must all be host arrays or all be device tensors")
        _cabi.check(self._lib.ba_set_observations(self._h, p_ptr, p_cam, p_xy, mems.pop(), self.stream))

    def set_observations_dense(self, x):
        """Dense ``x (N, M, 2)`` float64 exactly as the reference constructor receives it (one
        point-major or camera-major block, host array or CUDA tensor): no host-side copy."""
        if hasattr(x, "data_ptr") and getattr(x, "is_cuda", False):
            ptr, mem, strides = x.data_ptr(), _cabi.BA_MEM_DEVICE, tuple(x.stride())
        else:
            ptr, mem, strides = x.ctypes.data, _cabi.BA_MEM_HOST, tuple(s // 8 for s in x.strides)
        if tuple(x.shape) != (self.n_points, self.n_cams, 2) or strides[2] != 1:
            raise ValueError("x must be (n_points, n_cams, 2) with unit stride on the last axis")
        _cabi.check(self._lib.ba_set_observations_dense(self._h, ptr, strides[0], strides[1], mem, self.stream))

    def set_state(self, X=None, R=None, t=None, f=None, u=None):
        ptrs, mems, keep = [], set(), []
        for a in (X, R, t, f, u):
            p, m, k = _ptr(a, np.float64)
            ptrs.append(p)
            keep.append(k)
            if p is not None:
                mems.add(m)
        if len(mems) > 1:
            raise ValueError("state arrays must all be host arrays or all be device tensors")
        mem = mems.pop() if mems else _cabi.BA_MEM_HOST
        _cabi.check(self._lib.ba_set_state(self._h, *ptrs, mem, self.stream))

    def get_state(self, which: int = 0):
        N, M = self.n_points, self.n_cams
        X, R, t = np.empty((N, 3)), np.empty((M, 3, 3)), np.empty((M, 3))
        f, u = np.empty(M), np.empty((M, 2))
        _cabi.check(self._lib.ba_get_state(self._h, which, X.ctypes.data, R.ctypes.data, t.ctypes.data,
                                           f.ctypes.data, u.ctypes.data, _cabi.BA_MEM_HOST, self.stream))
        return X, R, t, f, u

    def set_state_global(self, X, R, t, f, u):
        """State in the caller's frame; the gauge normalisation (:208-240) runs on the device."""
        ptrs, mems, keep = [], set(), []
        for a in (X, R, t, f, u):
            p, m, k = _ptr(a, np.float64)
            ptrs.append(p)
            keep.append(k)
            mems.add(m)
        if len(mems) > 1:
            raise ValueError("state arrays must all be host arrays or all be device tensors")
        _cabi.check(self._lib.ba_set_state_global(self._h, *ptrs, mems.pop(), self.stream))

    def get_state_global(self, which: int = 0):
        """(X, K, R, t) back in the caller's frame (:242-258, :283-289), transformed on the device."""
        N, M = self.n_points, self.n_cams
        X, K, R, t = np.empty((N, 3)), np.empty((M, 3, 3)), np.empty((M, 3, 3)), np.empty((M, 3))
        _cabi.check(self._lib.ba_get_state_global(self._h, which, X.ctypes.data, K.ctypes.data, R.ctypes.data,
                                                  t.ctypes.data, _cabi.BA_MEM_HOST, self.stream))
        return X, K, R, t

    # -- single phases ------------------------------------------------------------------------
    def cost(self, which: int = 0) -> float:
        _cabi.check(self._lib.ba_cost(self._h, which, self.stream))
        return float(self.cost_values()[which])

    def cost_values(self) -> np.ndarray:
        return self.buffer("COST")

    def linearize(self):
        _cabi.check(self._lib.ba_linearize(self._h, self.stream))

    def build_reduced(self, c: float):
        _cabi.check(self._lib.ba_build_reduced(self._h, float(c), self.stream))

    def solve_trial(self, c: float):
        _cabi.check(self._lib.ba_solve_trial(self._h, float(c), self.stream))

    def covariance(self, points: bool = True):
        """(point_cov (N,3,3) or None, cam_cov (M,9,9), sigma2) at the current state, undamped, in the
        normalised frame and the parameter order (f, u0, v0, t, w); see ``ba_covariance``."""
        pc = np.empty((self.n_points, 3, 3)) if points else None
        cc = np.empty((self.n_cams, 9, 9))
        s2 = C.c_double()
        _cabi.check(self._lib.ba_covariance(self._h, None if pc is None else pc.ctypes.data, cc.ctypes.data,
                                            C.byref(s2), _cabi.BA_MEM_HOST, self.stream))
        return pc, cc, s2.value

    # -- LM loop ------------------------------------------------------------------------------
    def lm_begin(self, scale_factor, delta_tol, max_iter, max_retries=200):
        _cabi.check(self._lib.ba_lm_begin(self._h, float(scale_factor), float(delta_tol), int(max_iter),
                                          int(max_retries), self.stream))

    def lm_phase_reduce(self):
        _cabi.check(self._lib.ba_lm_phase_reduce(self._h, self.stream))

    def lm_phase_solve(self):
        _cabi.check(self._lib.ba_lm_phase_solve(self._h, self.stream))

    def lm_phase_decide(self):
        _cabi.check(self._lib.ba_lm_phase_decide(self._h, self.stream))

    def lm_state(self) -> _cabi.LMState:
        st = _cabi.LMState()
        _cabi.check(self._lib.ba_lm_state_get(self._h, C.byref(st), self.stream))
        return st

    def lm_state_post(self, slot: int) -> None:
        """Enqueue a copy of the control block into pinned slot 0/1 (no host synchronisation)."""
        _cabi.check(self._lib.ba_lm_state_post(self._h, int(slot), self.stream))

    def lm_state_wait(self, slot: int) -> _cabi.LMState:
        """Block until the copy posted into `slot` has landed and return it."""
        st = _cabi.LMState()
        _cabi.check(self._lib.ba_lm_state_wait(self._h, int(slot), C.byref(st)))
        return st

    def lm_iterate(self) -> _cabi.LMState:
        st = _cabi.LMState()
        _cabi.check(self._lib.ba_lm_iterate(self._h, C.byref(st), self.stream))
        return st

    def lm_records(self, max_records: int = 4096):
        recs = (_cabi.IterRecord * max_records)()
        n = C.c_int(0)
        _cabi.check(self._lib.ba_lm_records(self._h, recs, max_records, C.byref(n), self.stream))
        return [recs[i] for i in range(n.value)]

    def lm_run(self, scale_factor, delta_tol, max_iter, max_retries=200, max_records=4096):
        recs = (_cabi.IterRecord * max_records)()
        n = C.c_int(0)
        st = _cabi.LMState()
        status = self._lib.ba_lm_run(self._h, float(scale_factor), float(delta_tol), int(max_iter),
                                     int(max_retries), recs, max_records, C.byref(n), C.byref(st),
                                     self.stream)
        _cabi.check(status)
        return [recs[i] for i in range(n.value)], st

    # -- sharded runs: sums over NVLink peer memory ---------------------------------------------
    def comm_attach(self, dist, group=None) -> None:
        """Connect this engine with the engines of the other ranks of `group` (one process per
        GPU, all on one box): every rank exports its exchange window as a CUDA IPC handle, the
        handles are gathered over ``torch.distributed`` (plumbing only) and mapped.  Afterwards
        ``lm_begin`` / ``lm_phase_*`` / ``lm_iterate`` / ``lm_run`` sum the partial reduced
        system and the costs over the ranks inside the library (``csrc/comm_peer.cu``)."""
        import torch

        rank, world = dist.get_rank(group), dist.get_world_size(group)
        nb = _cabi.BA_COMM_HANDLE_BYTES
        handle = (C.c_ubyte * nb)()
        _cabi.check(self._lib.ba_comm_create(self._h, rank, world, handle))
        on_gpu = str(dist.get_backend(group)) == "nccl"
        dev = f"cuda:{self.device}" if on_gpu else "cpu"
        mine = torch.frombuffer(bytearray(handle), dtype=torch.uint8).to(dev)
        if on_gpu:
            gathered = torch.empty(world * nb, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(gathered, mine, group=group)
            blob = gathered.cpu().numpy().tobytes()
        else:
            parts = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(parts, mine, group=group)
            blob = b"".join(t.numpy().tobytes() for t in parts)
        _cabi.check(self._lib.ba_comm_connect(self._h, blob))
        # a new window must be mapped by every rank before anybody stores into it; recycled
        # windows (the usual case after the first engine of a shape) are mapped already
        if any(blob[r * nb + nb - 8] for r in range(world)):
            dist.barrier(group)
        self._comm = (dist, group)

    def comm_size(self) -> int:
        r, w = C.c_int(), C.c_int()
        _cabi.check(self._lib.ba_comm_world(self._h, C.byref(r), C.byref(w)))
        return w.value

    # -- buffers ------------------------------------------------------------------------------
    def _device_tensor(self, getter):
        import torch

        p, n = C.c_void_p(), C.c_int64()
        _cabi.check(getter(self._h, C.byref(p), C.byref(n)))
        return torch.as_tensor(_DeviceView(p.value, n.value), device=f"cuda:{self.device}")

    def reduce_tensor(self):
        """torch view of the partial reduced system (all-reduced by sharded runs)."""
        return self._device_tensor(self._lib.ba_reduce_buffer)

    def cost_tensor(self):
        """torch view of [cost of current/initial state, cost of trial state]."""
        return self._device_tensor(self._lib.ba_cost_buffer)

    def buffer(self, name: str) -> np.ndarray:
        bid = _cabi.BUFFERS[name]
        n = C.c_int64()
        _cabi.check(self._lib.ba_buffer_size(self._h, bid, C.byref(n)))
        out = np.empty(n.value)
        _cabi.check(self._lib.ba_buffer_read(self._h, bid, out.ctypes.data, n.value, self.stream))
        return out

    # -- profiling ----------------------------------------------------------------------------
    def profile_enable(self, on: bool = True):
        _cabi.check(self._lib.ba_profile_enable(self._h, 1 if on else 0))

    def profile_reset(self):
        _cabi.check(self._lib.ba_profile_reset(self._h))

    def matrix_free(self) -> bool:
        """Dense scene linearised matrix-free (Jacobian rows re-derived where they are used)."""
        return bool(self._lib.ba_matrix_free(self._h))

    def syrk_emulated(self) -> bool:
        """Dense Schur product on the INT8 tensor cores (Ozaki scheme II) rather than DMMA."""
        return bool(self._lib.ba_syrk_emulated(self._h))

    def profile(self) -> dict:
        out = {}
        for g in ("k1", "k2", "k3", "k4", "cost", "other", "syrk", "chol", "comm"):
            ms, n = C.c_double(), C.c_int64()
            _cabi.check(self._lib.ba_profile_get(self._h, g.encode(), C.byref(ms), C.byref(n)))
            out[g] = {"ms": ms.value, "launches": n.value}
        return out


def launch_count() -> int:
    return int(_cabi.load().ba_launch_count())


def fp64_peak(device: int = 0, dmma=True) -> float:
    """TFLOP/s of a register-resident loop: dmma=True DMMA.8x8x4, False DFMA, 2 both interleaved."""
    v = C.c_double()
    mode = int(dmma) if isinstance(dmma, int) and not isinstance(dmma, bool) and dmma >= 2 else (1 if dmma else 0)
    _cabi.check(_cabi.load().ba_fp64_peak(device, mode, C.byref(v)))
    return v.value


def syrk_emu_info(k_pad: int) -> tuple[list[int], int]:
    """Moduli of the INT8 emulation of the Schur product and the bits b kept per entry for k_pad rows."""
    lib = _cabi.load()
    n, b = C.c_int(), C.c_int()
    _cabi.check(lib.ba_syrk_emu_info(int(k_pad), None, C.byref(n), None))
    arr = (C.c_int32 * n.value)()
    _cabi.check(lib.ba_syrk_emu_info(int(k_pad), arr, C.byref(n), C.byref(b)))
    return list(arr), b.value


def syrk_feed() -> str:
    """Operand feed of the 128-tile SYRK kernel, which bench.py reports as `operand_feed`: always
    "tma" (cp.async.bulk.tensor + mbarriers), the only feed that kernel has."""
    return "tma"
