"""ctypes binding of libwdx_b200.so (C ABI in include/wdx_b200.h).

The CUDA library is the only compute path: if it cannot be loaded this module
raises — there is no CPU or PyTorch fallback behind it.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WDX_B200_LIB") or os.path.join(_HERE, "lib", "libwdx_b200.so")  # override: kernel-variant experiments

WDX_F64, WDX_F32 = 0, 1
MODE_EXACT_F64, MODE_FAST_F32, MODE_FAST_F32_GUARDED = 0, 1, 2
MODES = {"exact": MODE_EXACT_F64, "fast": MODE_FAST_F32, "guarded": MODE_FAST_F32_GUARDED}
FLAG_NONFINITE, FLAG_RECOMPUTED, FLAG_GUARD_OVERFLOW = 1, 2, 4

# every symbol include/wdx_b200.h declares
EXPORTS = [
    "wdx_model_create", "wdx_model_destroy", "wdx_model_set_guard", "wdx_model_set_chunk_reads", "wdx_model_set_sv_splits",
    "wdx_predict", "wdx_distance_matrix_to", "wdx_last_error", "wdx_device_count",
    "wdx_kernel_launch_count", "wdx_model_enable_timing", "wdx_model_last_kernel_ms", "wdx_model_last_kernel_ms_mode", "wdx_version",
    "wdx_fp_create", "wdx_fp_destroy", "wdx_fp_extract", "wdx_fp_extract_ex", "wdx_fp_set_consensus", "wdx_fp_predict", "wdx_fp_enable_timing", "wdx_fp_last_kernel_ms", "wdx_fp_set_long_slice_len", "wdx_fp_set_numpy1_promotion", "wdx_fp_set_resume_status",
    "wdx_cnn_create", "wdx_cnn_destroy", "wdx_cnn_detect", "wdx_cnn_prepare", "wdx_cnn_predict", "wdx_cnn_score_len", "wdx_cnn_set_guard", "wdx_cnn_enable_timing",
    "wdx_cnn_last_kernel_ms",
    "wdx_validate_create", "wdx_validate_destroy", "wdx_validate_run", "wdx_validate_enable_timing", "wdx_validate_last_kernel_ms", "wdx_validate_set_verdict_only", "wdx_validate_set_early", "wdx_validate_run_ex", "wdx_validate_run_report", "wdx_calibrate_rows", "wdx_validate_set_llr",
    "wdx_zstd_decompress", "wdx_vbz_decode_rows",
]

_lib = None
_lock = threading.Lock()


class WdxError(RuntimeError):
    pass


def load():
    """Load (building first if the sources are newer and nvcc is present)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        default_lib = "WDX_B200_LIB" not in os.environ
        if not os.path.exists(LIB_PATH):
            try:
                from . import build as _build

                _build.build()
            except Exception as e:  # noqa: BLE001
                raise WdxError(
                    f"libwdx_b200.so is not built ({LIB_PATH}) and could not be built here: {e}. "
                    "Run `python -m warpdemux_b200.build`. There is no CPU fallback."
                ) from e
        elif default_lib:
            # a library older than its sources would silently run old kernels: rebuild where nvcc is at hand, else say so
            from . import build as _build

            try:
                if _build.needs_build():
                    try:
                        _build._nvcc()
                    except RuntimeError:
                        import warnings

                        warnings.warn(f"{LIB_PATH} is older than warpdemux_b200/csrc (no nvcc here to rebuild it)", RuntimeWarning)
                    else:
                        _build.build()
            except OSError:
                pass
        try:
            L = C.CDLL(LIB_PATH)
        except OSError as e:
            raise WdxError(f"cannot load {LIB_PATH}: {e}. There is no CPU fallback.") from e
        vp, i32, i64, f64 = C.c_void_p, C.c_int, C.c_int64, C.c_double
        L.wdx_model_create.restype = i32
        L.wdx_model_create.argtypes = [vp, i32, i32, vp, i32, vp, vp, vp, vp, vp, vp, i32, f64, f64, i32, i32,
                                       C.POINTER(vp)]
        L.wdx_model_destroy.restype = None
        L.wdx_model_destroy.argtypes = [vp]
        L.wdx_model_set_guard.restype = i32
        L.wdx_model_set_guard.argtypes = [vp, f64]
        L.wdx_model_set_chunk_reads.restype = i32
        L.wdx_model_set_chunk_reads.argtypes = [vp, i64]
        L.wdx_model_set_sv_splits.restype = i32
        L.wdx_model_set_sv_splits.argtypes = [vp, i32]
        L.wdx_predict.restype = i32
        L.wdx_predict.argtypes = [vp, vp, i64, i32, i32, vp, vp, vp, vp, vp, vp]
        L.wdx_distance_matrix_to.restype = i32
        L.wdx_distance_matrix_to.argtypes = [vp, i64, vp, i64, i32, i32, f64, i32, vp, i32, i32, vp]
        L.wdx_last_error.restype = C.c_char_p
        L.wdx_device_count.restype = i32
        L.wdx_kernel_launch_count.restype = i64
        L.wdx_model_enable_timing.restype = i32
        L.wdx_model_enable_timing.argtypes = [vp, i32]
        L.wdx_model_last_kernel_ms.restype = i32
        L.wdx_model_last_kernel_ms.argtypes = [vp, C.POINTER(f64), C.POINTER(i32)]
        L.wdx_model_last_kernel_ms_mode.restype = i32
        L.wdx_model_last_kernel_ms_mode.argtypes = [vp, i32, C.POINTER(f64), C.POINTER(i32)]
        L.wdx_version.restype = C.c_char_p
        L.wdx_fp_create.restype = i32
        L.wdx_fp_create.argtypes = [vp, i32, C.POINTER(vp)]
        L.wdx_fp_destroy.restype = None
        L.wdx_fp_destroy.argtypes = [vp]
        L.wdx_fp_extract.restype = i32
        L.wdx_fp_extract.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]
        L.wdx_fp_extract_ex.restype = i32
        L.wdx_fp_extract_ex.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp]
        L.wdx_fp_set_long_slice_len.restype = i32
        L.wdx_fp_set_long_slice_len.argtypes = [vp, C.c_int32]
        L.wdx_fp_set_numpy1_promotion.restype = i32
        L.wdx_fp_set_numpy1_promotion.argtypes = [vp, i32]
        L.wdx_fp_set_resume_status.restype = i32
        L.wdx_fp_set_resume_status.argtypes = [vp, C.c_int32]
        L.wdx_fp_set_consensus.restype = i32
        L.wdx_fp_set_consensus.argtypes = [vp, vp]
        L.wdx_fp_predict.restype = i32
        L.wdx_fp_predict.argtypes = [vp, vp, vp, i64, i64, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp]
        L.wdx_fp_enable_timing.restype = i32
        L.wdx_fp_enable_timing.argtypes = [vp, i32]
        L.wdx_fp_last_kernel_ms.restype = i32
        L.wdx_fp_last_kernel_ms.argtypes = [vp, C.POINTER(f64), C.POINTER(i32)]
        L.wdx_cnn_create.restype = i32
        L.wdx_cnn_create.argtypes = [vp] + [vp] * 8 + [i32, C.POINTER(vp)]
        L.wdx_cnn_destroy.restype = None
        L.wdx_cnn_destroy.argtypes = [vp]
        L.wdx_cnn_detect.restype = i32
        L.wdx_cnn_detect.argtypes = [vp, vp, i64, i64, i32, vp, vp, vp, vp]
        L.wdx_cnn_prepare.restype = i32
        L.wdx_cnn_prepare.argtypes = [vp, vp, i64, i64, vp, vp]
        L.wdx_cnn_predict.restype = i32
        L.wdx_cnn_predict.argtypes = [vp, vp, i64, i32, i32, vp, vp, vp]
        L.wdx_cnn_score_len.restype = i32
        L.wdx_cnn_score_len.argtypes = [vp, i64, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.wdx_cnn_set_guard.restype = i32
        L.wdx_cnn_set_guard.argtypes = [vp, f64]
        L.wdx_cnn_enable_timing.restype = i32
        L.wdx_cnn_enable_timing.argtypes = [vp, i32]
        L.wdx_cnn_last_kernel_ms.restype = i32
        L.wdx_cnn_last_kernel_ms.argtypes = [vp, C.POINTER(f64), C.POINTER(i32)]
        L.wdx_validate_create.restype = i32
        L.wdx_validate_create.argtypes = [vp, i32, C.POINTER(vp)]
        L.wdx_validate_destroy.restype = None
        L.wdx_validate_destroy.argtypes = [vp]
        L.wdx_validate_run.restype = i32
        L.wdx_validate_run.argtypes = [vp, vp, i64, i64, vp, vp, i32, vp, vp, vp, vp, vp]
        L.wdx_validate_run_ex.restype = i32
        L.wdx_validate_run_ex.argtypes = [vp, vp, i64, i64, vp, vp, i32, vp, vp, vp, vp, vp, vp]
        L.wdx_validate_run_report.restype = i32
        L.wdx_validate_run_report.argtypes = [vp, vp, i64, i64, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp]
        L.wdx_calibrate_rows.restype = i32
        L.wdx_calibrate_rows.argtypes = [vp, i64, i64, vp, vp, vp, vp, i64, i32, vp]
        L.wdx_zstd_decompress.restype = i32
        L.wdx_zstd_decompress.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, i32, vp]
        L.wdx_vbz_decode_rows.restype = i32
        L.wdx_vbz_decode_rows.argtypes = [vp, vp, vp, i64, vp, i64, vp, vp, vp, i64, vp, vp, i32, vp]
        L.wdx_validate_set_verdict_only.restype = i32
        L.wdx_validate_set_verdict_only.argtypes = [vp, i32]
        L.wdx_validate_set_early.restype = i32
        L.wdx_validate_set_early.argtypes = [vp, vp, vp]
        L.wdx_validate_set_llr.restype = i32
        L.wdx_validate_set_llr.argtypes = [vp, vp]
        L.wdx_validate_enable_timing.restype = i32
        L.wdx_validate_enable_timing.argtypes = [vp, i32]
        L.wdx_validate_last_kernel_ms.restype = i32
        L.wdx_validate_last_kernel_ms.argtypes = [vp, C.POINTER(f64), C.POINTER(i32)]
        _lib = L
        return L


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().wdx_last_error().decode(errors="replace")
        if rc == -1:
            raise ValueError(f"{what}: {msg}")
        if rc == -3:
            raise MemoryError(f"{what}: {msg}")
        raise WdxError(f"{what}: {msg} (status {rc})")


def device_count() -> int:
    return int(load().wdx_device_count())


def kernel_launch_count() -> int:
    return int(load().wdx_kernel_launch_count())
