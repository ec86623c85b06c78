"""ctypes binding of the C ABI in include/tpls_b200.h.

The shared library ``libtpls_b200.so`` is built in-tree by
``cmtf_pls_b200/csrc/Makefile`` (``__graft_entry__.build()``).  There is no CPU
fallback: if the library is missing, or no sm_100 device is visible, using the
estimators raises.
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtpls_b200.so")

F32, F64 = 0, 1
X_MAY_OVERWRITE = 1
FIT_NORMALIZE_ON_BREAK = 1
FIT_PROFILE = 2
FIT_COVARIANCE = 4
MAX_TENSORS = 8
MAX_MODES = 8
E_BATCH_UNSUPPORTED = 2   # tpls_fit_batch: a problem is outside the batch kernel's limits, nothing was written

_lib = None


class TplsError(RuntimeError):
    pass


class Stats(C.Structure):
    _fields_ = [
        ("fit_ms", C.c_double),
        ("alg_bytes", C.c_double),
        ("streamed_bytes", C.c_double),
        ("kernel_launches", C.c_int64),
        ("total_trips", C.c_int64),
        ("collectives", C.c_int64),
        ("h2d_bytes", C.c_double),
        ("covariance_mode", C.c_int64),
        ("last_transform_path", C.c_int64),
        ("graph_launches", C.c_int64),
        ("launches_per_trip", C.c_int64),
        ("xchg_count", C.c_int64),
        ("xchg_ms", C.c_double),
        ("xchg_wait_ms", C.c_double),
        ("resident_loops", C.c_int64),
    ]


KERNEL_CLASSES = ["colstat", "contract", "project", "deflate_contract", "residual", "rank1", "yside", "other", "nccl", "xchg"]


class Profile(C.Structure):
    _fields_ = [("ms", C.c_double * 10), ("launches", C.c_int64 * 10), ("bytes", C.c_double * 10)]


class BatchOut(C.Structure):
    """Mirror of ``tpls_batch_out``: caller-owned results of ``tpls_fit_batch``, leading axis = problem."""
    _fields_ = [
        ("T", C.c_void_p),
        ("U", C.c_void_p),
        ("Q", C.c_void_p),
        ("W", C.c_void_p * MAX_TENSORS),
        ("coef", C.c_void_p),
        ("r2x", C.c_void_p),
        ("r2y", C.c_void_p),
        ("x_mean", C.c_void_p * MAX_TENSORS),
        ("y_mean", C.c_void_p),
        ("trips", C.c_void_p),
        ("converged", C.c_void_p),
        ("has_missing", C.c_void_p),
        ("fit_ms", C.c_double),
    ]


# name -> (restype, argtypes); every symbol declared in include/tpls_b200.h
_H = C.c_void_p
_P = C.c_void_p
SIGNATURES = {
    "tpls_version": (C.c_int, []),
    "tpls_last_error": (C.c_char_p, [_H]),
    "tpls_create": (C.c_int, [C.POINTER(_H), C.c_int, _P]),
    "tpls_destroy": (C.c_int, [_H]),
    "tpls_set_stream": (C.c_int, [_H, _P]),
    "tpls_comm_unique_id": (C.c_int, [_P]),
    "tpls_comm_init": (C.c_int, [_H, _P, C.c_int, C.c_int]),
    "tpls_comm_xchg_handle": (C.c_int, [_H, _P]),
    "tpls_comm_xchg_open": (C.c_int, [_H, _P]),
    "tpls_set_x": (C.c_int, [_H, C.c_int, _P, C.c_int, C.c_int, C.POINTER(C.c_int64), C.c_int]),
    "tpls_set_y": (C.c_int, [_H, _P, C.c_int64, C.c_int64]),
    "tpls_set_row_weights": (C.c_int, [_H, _P, C.c_int64]),
    "tpls_fit": (C.c_int, [_H, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int]),
    "tpls_get_x_factor": (C.c_int, [_H, C.c_int, C.c_int, _P]),
    "tpls_get_y_factor": (C.c_int, [_H, C.c_int, _P]),
    "tpls_get_coef": (C.c_int, [_H, _P]),
    "tpls_get_r2x": (C.c_int, [_H, C.c_int, _P]),
    "tpls_get_r2y": (C.c_int, [_H, _P]),
    "tpls_get_x_mean": (C.c_int, [_H, C.c_int, _P]),
    "tpls_get_y_mean": (C.c_int, [_H, _P]),
    "tpls_get_has_missing": (C.c_int, [_H, C.c_int, C.POINTER(C.c_int)]),
    "tpls_get_trips": (C.c_int, [_H, _P]),
    "tpls_get_converged": (C.c_int, [_H, _P]),
    "tpls_get_stats": (C.c_int, [_H, C.POINTER(Stats)]),
    "tpls_get_profile": (C.c_int, [_H, C.POINTER(Profile)]),
    "tpls_release_data": (C.c_int, [_H]),
    "tpls_trim": (C.c_int, [_H]),
    "tpls_transform": (C.c_int, [_H, C.c_int, C.c_int, C.POINTER(_P), C.POINTER(C.c_int), C.c_int64,
                                 C.POINTER(C.c_int64), C.POINTER(_P), C.POINTER(_P), _P, _P, _P]),
    "tpls_reconstruct": (C.c_int, [_H, C.c_int, _P, C.c_int64, C.c_int64, _P, _P, C.c_int, _P]),
    "tpls_fit_batch": (C.c_int, [_H, C.c_int, C.c_int64, C.POINTER(_P), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                 C.POINTER(C.POINTER(C.c_int64)), C.POINTER(C.c_int64), _P, C.c_int64, C.c_int64, _P,
                                 C.c_int, C.c_double, C.c_int, C.c_int, C.POINTER(BatchOut)]),
    "tpls_op_contract": (C.c_int, [_H, _P, C.c_int, C.c_int64, C.c_int64, _P, C.c_int, _P, C.POINTER(C.c_float), C.c_int]),
    "tpls_op_project": (C.c_int, [_H, _P, C.c_int, C.c_int64, C.c_int64, _P, C.c_int, _P, C.POINTER(C.c_float), C.c_int]),
    "tpls_op_deflate_contract": (C.c_int, [_H, _P, C.c_int, C.c_int64, C.c_int64, _P, _P, _P, C.c_int, _P, _P,
                                           C.POINTER(C.c_float), C.c_int]),
    "tpls_op_rank1": (C.c_int, [_H, _P, C.c_int, C.POINTER(C.c_int), C.c_double, C.c_int, _P, _P, C.POINTER(C.c_int),
                                C.POINTER(C.c_float), C.c_int]),
}


def load_library(path: str | None = None):
    """dlopen the C-ABI library and bind every declared symbol (no GPU needed)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("TPLS_B200_LIB") or LIB_PATH   # TPLS_B200_LIB: another build of the library (A/B runs)
    if not os.path.exists(p):
        raise TplsError(
            f"{p} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C cmtf_pls_b200/csrc).  cmtf_pls_b200 has no CPU fallback.")
    lib = C.CDLL(p, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def _ptr(a) -> int:
    """Raw address of a numpy array (host) or torch tensor (host or CUDA)."""
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return int(a.data_ptr())


def dtype_code(a) -> int:
    name = str(a.dtype).replace("torch.", "")
    if name == "float32":
        return F32
    if name == "float64":
        return F64
    raise TypeError(f"X must be float32 or float64, got {a.dtype}")


class Engine:
    """One fit context (``tpls_handle``) on one CUDA device."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self.lib = load_library()
        self.h = _H()
        rc = self.lib.tpls_create(C.byref(self.h), int(device), C.c_void_p(stream) if stream else None)
        if rc != 0:
            raise TplsError(self.lib.tpls_last_error(None).decode())
        self.device = device
        self._keep = []
        self._stream = stream or 0
        self.comm_key = None      # (id of the process group, rank, world) the handle's communicator belongs to
        self.comm_world = 1
        self.exchange = "none"    # "peer" (CUDA IPC exchange kernels), "nccl", or "none" (single GPU)

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.tpls_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise TplsError(self.lib.tpls_last_error(self.h).decode())

    def set_stream(self, stream: int):
        """Follow the caller's current CUDA stream (0: the handle's private stream)."""
        if stream != self._stream:
            self._ck(self.lib.tpls_set_stream(self.h, C.c_void_p(stream) if stream else None))
            self._stream = stream

    # ---- multi-GPU ----
    def unique_id(self) -> bytes:
        buf = C.create_string_buffer(128)
        if self.lib.tpls_comm_unique_id(buf) != 0:
            raise TplsError(self.lib.tpls_last_error(None).decode())
        return buf.raw

    def init_comm(self, uid: bytes, rank: int, world: int):
        self._ck(self.lib.tpls_comm_init(self.h, C.c_char_p(uid), rank, world))

    def xchg_handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        self._ck(self.lib.tpls_comm_xchg_handle(self.h, buf))
        return buf.raw

    def xchg_open(self, handles):
        """handles: list of the ranks' 64-byte IPC handles in rank order, or None to switch the exchange off."""
        arg = None if handles is None else C.c_char_p(b"".join(handles))
        self._ck(self.lib.tpls_comm_xchg_open(self.h, arg))

    # ---- data ----
    def set_x(self, index, x, flags=0):
        shape = (C.c_int64 * len(x.shape))(*[int(s) for s in x.shape])
        self._keep.append(x)
        self._ck(self.lib.tpls_set_x(self.h, index, _ptr(x), dtype_code(x), len(x.shape), shape, flags))

    def set_y(self, y):
        self._keep.append(y)
        self._ck(self.lib.tpls_set_y(self.h, _ptr(y), int(y.shape[0]), int(y.shape[1])))

    def set_row_weights(self, w):
        if w is None:
            self._ck(self.lib.tpls_set_row_weights(self.h, None, 0))
            return
        self._keep.append(w)
        self._ck(self.lib.tpls_set_row_weights(self.h, _ptr(w), int(w.shape[0])))

    def fit(self, n_tensors, n_components, tol, max_iter, flags=0):
        try:
            self._ck(self.lib.tpls_fit(self.h, n_tensors, n_components, float(tol), int(max_iter), flags))
        finally:
            self._keep.clear()   # the staged inputs are not pinned by a failed fit either

    def fit_batch(self, batch, xs, x_strides, shapes, y, y_stride, m, row_w, n_components, tol, max_iter, out, flags=0):
        """tpls_fit_batch.  xs / y / row_w: numpy arrays or torch tensors (host or CUDA) with the problems at the
        given element strides; ``shapes`` the per-problem shapes (n, d1, ...); ``out`` a filled BatchOut.  Returns
        True when the batch kernel ran, False on E_BATCH_UNSUPPORTED (nothing written); raises on errors."""
        L = len(xs)
        ptrs = (_P * L)(*[_ptr(x) for x in xs])
        dts = (C.c_int * L)(*[dtype_code(x) for x in xs])
        nds = (C.c_int * L)(*[len(s) for s in shapes])
        shp = [(C.c_int64 * len(s))(*[int(v) for v in s]) for s in shapes]
        shps = (C.POINTER(C.c_int64) * L)(*[C.cast(a, C.POINTER(C.c_int64)) for a in shp])
        strd = (C.c_int64 * L)(*[int(v) for v in x_strides])
        rc = self.lib.tpls_fit_batch(self.h, L, int(batch), ptrs, dts, nds, shps, strd,
                                     _ptr(y), int(m), int(y_stride), None if row_w is None else _ptr(row_w),
                                     int(n_components), float(tol), int(max_iter), int(flags), C.byref(out))
        if rc == E_BATCH_UNSUPPORTED:
            return False
        self._ck(rc)
        return True

    # ---- results ----
    def _host_out(self, rows, cols):
        """Host array for a device result.  Large ones (the N x R score matrices) are backed by pinned memory
        from torch's caching host allocator once this engine is seen to fit REPEATEDLY (cross-validation sweeps,
        bootstraps, benchmarks): the device-to-host copy then runs at DMA speed instead of through the driver's
        bounce buffers (160 MB of scores: ~4 ms instead of ~45 ms).  Pinning fresh memory costs more than that,
        so the first fit of a process stays on pageable memory and never pays for it.  The ndarray keeps the
        pinned tensor alive; its block returns to torch's cache when the array is garbage-collected.
        TPLS_PAGEABLE_OUT=1 turns this off."""
        if rows * cols * 8 >= (1 << 22):
            self._big_fetches = getattr(self, "_big_fetches", 0) + 1
            if self._big_fetches > 2 and os.environ.get("TPLS_PAGEABLE_OUT", "") == "":
                try:
                    import torch
                    return torch.empty((rows, cols), dtype=torch.float64, pin_memory=True).numpy()
                except Exception:  # noqa: BLE001 -- no torch / pinning refused: pageable memory works too
                    pass
        return np.empty((rows, cols), dtype=np.float64)

    def x_factor(self, index, mode, rows, R):
        out = self._host_out(rows, R)
        self._ck(self.lib.tpls_get_x_factor(self.h, index, mode, out.ctypes.data))
        return out

    def y_factor(self, which, rows, R):
        out = self._host_out(rows, R)
        self._ck(self.lib.tpls_get_y_factor(self.h, which, out.ctypes.data))
        return out

    def coef(self, R):
        out = np.empty((R, R), dtype=np.float64)
        self._ck(self.lib.tpls_get_coef(self.h, out.ctypes.data))
        return out

    def r2x(self, index, R):
        out = np.empty(R, dtype=np.float64)
        self._ck(self.lib.tpls_get_r2x(self.h, index, out.ctypes.data))
        return out

    def r2y(self, R):
        out = np.empty(R, dtype=np.float64)
        self._ck(self.lib.tpls_get_r2y(self.h, out.ctypes.data))
        return out

    def x_mean(self, index, shape, dtype):
        out = np.empty(shape, dtype=dtype)
        self._ck(self.lib.tpls_get_x_mean(self.h, index, out.ctypes.data))
        return out

    def y_mean(self, m):
        out = np.empty(m, dtype=np.float64)
        self._ck(self.lib.tpls_get_y_mean(self.h, out.ctypes.data))
        return out

    def has_missing(self, index) -> bool:
        v = C.c_int(0)
        self._ck(self.lib.tpls_get_has_missing(self.h, index, C.byref(v)))
        return bool(v.value)

    def trips(self, R):
        out = np.empty(R, dtype=np.int32)
        self._ck(self.lib.tpls_get_trips(self.h, out.ctypes.data))
        return out

    def converged(self, R):
        out = np.empty(R, dtype=np.int32)
        self._ck(self.lib.tpls_get_converged(self.h, out.ctypes.data))
        return out.astype(bool)

    def stats(self) -> dict:
        s = Stats()
        self._ck(self.lib.tpls_get_stats(self.h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in Stats._fields_}

    def profile(self) -> dict:
        p = Profile()
        self._ck(self.lib.tpls_get_profile(self.h, C.byref(p)))
        return {k: dict(ms=p.ms[i], launches=p.launches[i], bytes=p.bytes[i]) for i, k in enumerate(KERNEL_CLASSES)}

    def trim(self):
        self._ck(self.lib.tpls_trim(self.h))

    def release_data(self):
        self._ck(self.lib.tpls_release_data(self.h))

    def reconstruct(self, scores, wkron, mean):
        """(n, p) float64: mean + scores @ wkron, formed on the device (tpls.py:188-189)."""
        scores = np.ascontiguousarray(scores, dtype=np.float64)
        wkron = np.ascontiguousarray(wkron, dtype=np.float64)
        n, R = scores.shape
        p = wkron.shape[1]
        out = self._host_out(n, p)
        mp, md = (None, 0) if mean is None else (mean.ctypes.data, dtype_code(mean))
        self._ck(self.lib.tpls_reconstruct(self.h, R, scores.ctypes.data, n, p, wkron.ctypes.data, mp, md, out.ctypes.data))
        return out

    def transform(self, xs, means, wkrons, proj_offset=None, proj_gram=None):
        """xs[l]: (n_new, ...) array/tensor; means[l]: numpy, X's dtype; wkrons[l]: (R, P) float64 numpy;
        proj_offset (R,), proj_gram (R, R): constants of the read-only path for complete data (or None)."""
        L = len(xs)
        n_new = int(xs[0].shape[0])
        R = int(wkrons[0].shape[0])
        xp = (_P * L)(*[_ptr(x) for x in xs])
        dt = (C.c_int * L)(*[dtype_code(x) for x in xs])
        ps = (C.c_int64 * L)(*[int(w.shape[1]) for w in wkrons])
        mp = (_P * L)(*[_ptr(m) for m in means])
        wp = (_P * L)(*[_ptr(w) for w in wkrons])
        out = self._host_out(n_new, R)
        po = None if proj_offset is None else proj_offset.ctypes.data
        pgm = None if proj_gram is None else proj_gram.ctypes.data
        self._ck(self.lib.tpls_transform(self.h, L, R, xp, dt, n_new, ps, mp, wp, po, pgm, out.ctypes.data))
        return out
