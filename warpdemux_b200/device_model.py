"""Device-resident model handle: thin owner of a `wdx_model*` (include/wdx_b200.h)."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import numpy as np

from . import _lib
from .model_io import ModelParams


def _ptr(a) -> Optional[int]:
    """Address of a numpy array, a torch tensor (host or CUDA) or a raw int."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return int(a.data_ptr())
    raise TypeError(f"cannot take the address of {type(a)}")


class DeviceModel:
    """One model replica on one GPU.  Not picklable by design — the picklable
    object is `warpdemux_b200.models.dtw_svm.DTW_SVM`, which creates this lazily
    in whichever process ends up calling `predict`."""

    def __init__(self, params: ModelParams, device: int = 0):
        self.params = params
        self.device = int(device)
        lib = _lib.load()
        h = C.c_void_p()
        p = params
        rc = lib.wdx_model_create(
            p.sv.ctypes.data, p.n_sv, p.L, p.n_sv_class.ctypes.data, p.k, p.dual_coef.ctypes.data,
            p.rho.ctypes.data, p.probA.ctypes.data, p.probB.ctypes.data, p.thresholds.ctypes.data,
            p.label_map.ctypes.data, int(p.window or 0), float(p.penalty or 0.0), float(p.gamma),
            int(p.pwr_dist), self.device, C.byref(h))
        _lib.check(rc, "wdx_model_create")
        self._h = h
        self.thresholds = p.thresholds   # the array uploaded; a holder of `params` rebuilds when it is replaced

    def close(self):
        if getattr(self, "_h", None):
            _lib.load().wdx_model_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def set_guard(self, guard: float):
        _lib.check(_lib.load().wdx_model_set_guard(self._h, float(guard)), "wdx_model_set_guard")

    def set_chunk_reads(self, n: int):
        _lib.check(_lib.load().wdx_model_set_chunk_reads(self._h, int(n)), "wdx_model_set_chunk_reads")

    def set_sv_splits(self, splits: int):
        _lib.check(_lib.load().wdx_model_set_sv_splits(self._h, int(splits)), "wdx_model_set_sv_splits")

    def enable_timing(self, on: bool = True):
        _lib.check(_lib.load().wdx_model_enable_timing(self._h, int(on)), "wdx_model_enable_timing")

    def last_kernel_ms(self) -> Tuple[float, int]:
        ms, n = C.c_double(), C.c_int()
        _lib.check(_lib.load().wdx_model_last_kernel_ms(self._h, C.byref(ms), C.byref(n)), "wdx_model_last_kernel_ms")
        return ms.value, n.value

    def last_kernel_ms_mode(self, exact: bool) -> Tuple[float, int]:
        ms, n = C.c_double(), C.c_int()
        _lib.check(_lib.load().wdx_model_last_kernel_ms_mode(self._h, int(exact), C.byref(ms), C.byref(n)),
                   "wdx_model_last_kernel_ms_mode")
        return ms.value, n.value

    def predict_raw(self, X, n: int, x_dtype: int, mode: int, labels, conf=None, prob=None, flags=None,
                    dist=None, stream: int = 0) -> None:
        """Pointer-level call: every buffer may be a numpy array, a torch tensor
        (CPU or CUDA) or an address."""
        rc = _lib.load().wdx_predict(self._h, _ptr(X), int(n), int(x_dtype), int(mode), _ptr(labels), _ptr(conf),
                                     _ptr(prob), _ptr(flags), _ptr(dist), stream or None)
        _lib.check(rc, "wdx_predict")

    def predict(self, X: np.ndarray, mode: str = "exact", want_dist: bool = False):
        """numpy in, numpy out: (labels int64[n], prob f64[n,k], conf f64[n], flags u8[n][, dist f32[n,n_sv]])."""
        X = np.asarray(X)
        if X.dtype == np.float32:
            xd = _lib.WDX_F32
        else:
            X = X.astype(np.float64, copy=False)
            xd = _lib.WDX_F64
        X = np.ascontiguousarray(X)
        n = X.shape[0]
        k = self.params.k
        labels = np.empty(n, dtype=np.int64)
        conf = np.empty(n, dtype=np.float64)
        prob = np.empty((n, k), dtype=np.float64)
        flags = np.zeros(n, dtype=np.uint8)
        dist = np.empty((n, self.params.n_sv), dtype=np.float32) if want_dist else None
        if n:
            self.predict_raw(X, n, xd, _lib.MODES[mode], labels, conf, prob, flags, dist)
            over = np.flatnonzero(flags & _lib.FLAG_GUARD_OVERFLOW)
            if over.size:
                # GUARDED: the device-side list of boundary reads was full; finish the
                # guarantee here by re-running exactly those reads in EXACT_F64.
                Xo = np.ascontiguousarray(X[over])
                lo, co = np.empty(over.size, np.int64), np.empty(over.size, np.float64)
                po, fo = np.empty((over.size, k), np.float64), np.zeros(over.size, np.uint8)
                self.predict_raw(Xo, over.size, xd, _lib.MODE_EXACT_F64, lo, co, po, fo, None)
                labels[over], conf[over], prob[over] = lo, co, po
                flags[over] = fo | _lib.FLAG_RECOMPUTED
        if want_dist:
            return labels, prob, conf, flags, dist
        return labels, prob, conf, flags


def distance_matrix(X: np.ndarray, Y: np.ndarray, window, penalty, mode: str = "exact",
                    out_dtype=np.float32, device: int = 0) -> np.ndarray:
    X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
    Y = np.ascontiguousarray(np.atleast_2d(Y), dtype=np.float64)
    if X.shape[1] != Y.shape[1]:
        raise ValueError("X and Y must have the same number of columns")
    out = np.empty((X.shape[0], Y.shape[0]), dtype=out_dtype)
    od = _lib.WDX_F32 if out.dtype == np.float32 else _lib.WDX_F64
    rc = _lib.load().wdx_distance_matrix_to(X.ctypes.data, X.shape[0], Y.ctypes.data, Y.shape[0], X.shape[1],
                                            int(window or 0), float(penalty or 0.0), _lib.MODES[mode],
                                            out.ctypes.data, od, int(device), None)
    _lib.check(rc, "wdx_distance_matrix_to")
    return out
