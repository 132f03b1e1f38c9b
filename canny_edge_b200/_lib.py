"""ctypes binding of libcanny_b200.so (the C ABI declared in include/canny_b200.h).

The library is hand-written sm_100a CUDA; there is no Python or CPU implementation behind these
calls.  Importing this module never needs a GPU (symbols can be inspected on a CPU box); calling a
compute entry point without a B200 raises CannyB200Error.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libcanny_b200.so"

OK, ERR_INVALID_ARG, ERR_NO_DEVICE, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOMEM = range(6)
MAX_RADIUS = 48


class CannyB200Error(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"libcanny_b200 status {status}: {message}")
        self.status = status


class BandRecord(C.Structure):
    _fields_ = [("label", C.c_int32), ("flags", C.c_int32)]


class Frame(C.Structure):
    """b200_frame: one frame of a b200_canny_frames_device list (device pointers, byte pitches)."""
    _fields_ = [("in_", C.c_void_p), ("in_row_pitch", C.c_int64), ("out", C.c_void_p), ("out_row_pitch", C.c_int64),
                ("height", C.c_int32), ("width", C.c_int32)]


_u8p, _i16p, _f32p = C.c_void_p, C.c_void_p, C.c_void_p  # raw addresses (numpy .ctypes.data / tensor.data_ptr())
_ctx = C.c_void_p

# name -> (restype, argtypes); must list EVERY function include/canny_b200.h declares
SIGNATURES = {
    "b200_version": (C.c_int, []),
    "b200_last_error": (C.c_char_p, []),
    "b200_ctx_create": (C.c_int, [C.c_int, C.POINTER(_ctx)]),
    "b200_ctx_destroy": (C.c_int, [_ctx]),
    "b200_ctx_set_stream": (C.c_int, [_ctx, C.c_void_p]),
    "b200_ctx_synchronize": (C.c_int, [_ctx]),
    "b200_ctx_set_chunk_frames": (C.c_int, [_ctx, C.c_int]),
    "b200_ctx_kernel_launches": (C.c_longlong, [_ctx]),
    "b200_ctx_transfer_bytes": (C.c_int, [_ctx, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]),
    "b200_ctx_front_kernel_stats": (C.c_int, [_ctx, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    "b200_host_bind_numa": (C.c_int, [C.c_int, C.POINTER(C.c_int)]),
    "b200_gaussian_window": (C.c_int, [C.c_float]),
    "b200_gaussian_kernel": (C.c_int, [C.c_float, _f32p, C.POINTER(C.c_int)]),
    "b200_direction_host": (C.c_int, [C.c_int, C.c_int]),
    "b200_isqrt_host": (C.c_int, [C.c_int]),
    "b200_gaussian": (C.c_int, [_ctx, _u8p, C.c_float, C.c_int, C.c_int, _i16p]),
    "b200_xy_gradient": (C.c_int, [_ctx, _i16p, C.c_int, C.c_int, _i16p, _i16p]),
    "b200_sobel": (C.c_int, [_ctx, _i16p, C.c_int, C.c_int, _i16p, _i16p]),
    "b200_nonmaximal": (C.c_int, [_ctx, _i16p, _i16p, C.c_int, C.c_int, _i16p]),
    "b200_hysteresis": (C.c_int, [_ctx, _i16p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "b200_canny": (C.c_int, [_ctx, _u8p, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, _i16p]),
    "b200_canny_steps": (C.c_int, [_ctx, _u8p, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, _i16p, _i16p, _i16p, _i16p, _i16p]),
    "b200_canny_bgr": (C.c_int, [_ctx, _u8p, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, _u8p, _i16p]),
    "b200_bgr_to_gray_device": (C.c_int, [_ctx, _u8p, C.c_size_t, _u8p]),
    "b200_canny_batch_host": (C.c_int, [_ctx, _u8p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, _u8p]),
    "b200_canny_batch_host_packed": (C.c_int, [_ctx, _u8p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_void_p]),
    "b200_canny_batch_device": (C.c_int, [_ctx, _u8p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, _u8p]),
    "b200_canny_batch_device_bgr": (C.c_int, [_ctx, _u8p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, _u8p]),
    "b200_canny_batch_device_strided": (C.c_int, [_ctx, _u8p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int,
                                                  C.c_int, _u8p, C.c_int64, C.c_int64]),
    "b200_canny_batch_device_bgr_strided": (C.c_int, [_ctx, _u8p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int,
                                                      C.c_int, _u8p, C.c_int64, C.c_int64]),
    "b200_cv_canny_device_strided": (C.c_int, [_ctx, _u8p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                                               C.c_double, C.c_int, _u8p, C.c_int64, C.c_int64]),
    "b200_cv_canny_aperture_device_strided": (C.c_int, [_ctx, _u8p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int,
                                                        C.c_double, C.c_double, C.c_int, C.c_int, _u8p, C.c_int64, C.c_int64]),
    "b200_canny_frames_device": (C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_int]),
    "b200_canny_frames_device_bgr": (C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_int]),
    "b200_cv_canny_frames_device": (C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int]),
    "b200_cv_canny_aperture_frames_device": (C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int]),
    "b200_cv_gaussian_canny_device_strided": (C.c_int, [_ctx, _u8p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int,
                                                        C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int,
                                                        C.c_int, _u8p, C.c_int64, C.c_int64]),
    "b200_cv_gaussian_canny_frames_device": (C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double,
                                                       C.c_double, C.c_double, C.c_int, C.c_int]),
    "b200_cv_gaussian_kernel": (C.c_int, [C.c_int, C.c_double, C.POINTER(C.c_int), C.POINTER(C.c_int32)]),
    "b200_profile_stages_device": (C.c_int, [_ctx, _u8p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, _u8p, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "b200_profile_pipeline_device": (C.c_int, [_ctx, _u8p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, _u8p, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "b200_hash_edges_device": (C.c_int, [_ctx, _u8p, C.c_size_t, C.c_ulonglong, C.POINTER(C.c_ulonglong)]),
    "b200_band_halo_rows": (C.c_int, [C.c_float]),
    "b200_band_record_count": (C.c_int, [C.c_int]),
    "b200_band_front": (C.c_int, [_ctx, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, _u8p]),
    "b200_band_boundary_export": (C.c_int, [_ctx, C.c_int, C.c_int, C.c_void_p]),
    "b200_band_finalize": (C.c_int, [_ctx, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _u8p]),
    "b200_bands_unique_id": (C.c_int, [C.c_void_p]),
    "b200_bands_create": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "b200_bands_create_group": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "b200_bands_destroy": (C.c_int, [C.c_void_p]),
    "b200_bands_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "b200_bands_input": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "b200_bands_run": (C.c_int, [C.c_void_p, _u8p]),
    "b200_bands_run_group": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p)]),
    "b200_bands_begin": (C.c_int, [C.c_void_p, _u8p]),
    "b200_bands_front": (C.c_int, [C.c_void_p]),
    "b200_bands_finish": (C.c_int, [C.c_void_p]),
    "b200_bands_check": (C.c_int, [C.c_void_p]),
    "b200_bands_set_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "b200_bands_stage_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "b200_synth_host": (C.c_int, [_u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int]),
    "b200_synth_device": (C.c_int, [_ctx, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int]),
    "b200_synth_rows_host": (C.c_int, [_u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int]),
    "b200_synth_rows_device": (C.c_int, [_ctx, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int]),
    "b200_direction_table_host": (C.c_int, [C.c_int, C.c_void_p]),
    "b200_direction_table_device": (C.c_int, [_ctx, C.c_int, C.c_void_p]),
    "b200_isqrt_table_device": (C.c_int, [_ctx, C.c_int, C.c_void_p]),
    "b200_division_check_device": (C.c_int, [_ctx, C.c_float, C.POINTER(C.c_ulonglong)]),
    "b200_division_mode_device": (C.c_int, [_ctx, C.c_float, C.POINTER(C.c_int)]),
    "b200_count_edges_device": (C.c_int, [_ctx, _u8p, C.c_size_t, C.POINTER(C.c_ulonglong)]),
    "b200_pack_edges_device": (C.c_int, [_ctx, _u8p, C.c_size_t, C.c_void_p]),
    "b200_unpack_edges_host": (C.c_int, [_u8p, C.c_size_t, C.c_void_p, C.c_int, C.c_int]),
    "b200_device_alloc": (C.c_int, [_ctx, C.c_size_t, C.POINTER(C.c_void_p)]),
    "b200_device_free": (C.c_int, [_ctx, C.c_void_p]),
    "b200_memcpy_h2d": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_size_t]),
    "b200_memcpy_d2h": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_size_t]),
    "b200_host_alloc_pinned": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "b200_host_free_pinned": (C.c_int, [C.c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Loads the in-tree shared library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m canny_edge_b200.build` "
            "(needs nvcc; there is no CPU implementation to fall back to)")
    lib = C.CDLL(str(LIB_PATH), mode=getattr(os, "RTLD_NOW", 2))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means header and library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != OK:
        msg = load().b200_last_error()
        raise CannyB200Error(status, msg.decode() if msg else "")
