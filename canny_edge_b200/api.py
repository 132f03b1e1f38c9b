"""Host-side mirror of the reference's stage API over the C ABI (numpy in, numpy out).

Function names and argument order follow the reference's GPU header src/cuda.h:4-10 and its CPU twin
src/utils.h:8-22 (`cuda_nonmaixmal_suppression` keeps the reference's spelling — it is the symbol
name).  Where the reference allocates its result with new[] and hands it back through a
reference-to-pointer, these return a fresh numpy array.  Every call runs the sm_100a kernels in
libcanny_b200.so; nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import numpy as np

from . import _lib
from ._lib import CannyB200Error, check, load

PI = 3.1415926535  # src/utils.h:4
EDGE = 255         # src/utils.h:5
NOEDGE = 0         # src/utils.h:6


def _ptr(a: np.ndarray) -> int:
    return a.ctypes.data


def _img(a, dtype) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=dtype)
    if a.ndim != 2:
        raise ValueError("expected a 2-D (height, width) array")
    return a


class Context:
    """Owns a b200_ctx: device, streams, workspace pool, cached Gaussian tables."""

    def __init__(self, device: int = 0):
        self._lib = load()
        h = C.c_void_p()
        check(self._lib.b200_ctx_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    def set_stream(self, cuda_stream: int) -> None:
        check(self._lib.b200_ctx_set_stream(self._h, C.c_void_p(cuda_stream)))

    def set_chunk_frames(self, frames: int) -> None:
        check(self._lib.b200_ctx_set_chunk_frames(self._h, int(frames)))

    def synchronize(self) -> None:
        check(self._lib.b200_ctx_synchronize(self._h))

    @property
    def kernel_launches(self) -> int:
        return int(self._lib.b200_ctx_kernel_launches(self._h))

    def front_kernel_stats(self):
        """(launches of the specialised front kernels, launches of the generic one) so far."""
        fast, gen = C.c_longlong(), C.c_longlong()
        check(self._lib.b200_ctx_front_kernel_stats(self._h, C.byref(fast), C.byref(gen)))
        return int(fast.value), int(gen.value)

    def close(self) -> None:
        if self._h:
            self._lib.b200_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def _h(ctx: Optional[Context]):
    return ctx.handle if ctx is not None else None


# ---------------------------------------------------------------------------------------------------
# host-side helpers
# ---------------------------------------------------------------------------------------------------
def createGaussianKernel(sigma: float) -> Tuple[np.ndarray, int]:
    """createGaussianKernel (src/utils.cpp:77-95): returns (kernel float32[window], window)."""
    lib = load()
    n = lib.b200_gaussian_window(C.c_float(sigma))
    if n <= 0:
        raise ValueError("sigma must be positive")
    w = np.zeros(n, np.float32)
    win = C.c_int()
    check(lib.b200_gaussian_kernel(C.c_float(sigma), _ptr(w), C.byref(win)))
    return w, win.value


# ---------------------------------------------------------------------------------------------------
# stage API (src/cuda.h:4-10)
# ---------------------------------------------------------------------------------------------------
def cuda_gaussian(img, sigma: float, ctx: Optional[Context] = None) -> np.ndarray:
    a = _img(img, np.uint8)
    out = np.empty(a.shape, np.int16)
    check(load().b200_gaussian(_h(ctx), _ptr(a), C.c_float(sigma), a.shape[0], a.shape[1], _ptr(out)))
    return out


def calculateXYGradient(blur, ctx: Optional[Context] = None) -> Tuple[np.ndarray, np.ndarray]:
    a = _img(blur, np.int16)
    gx, gy = np.empty(a.shape, np.int16), np.empty(a.shape, np.int16)
    check(load().b200_xy_gradient(_h(ctx), _ptr(a), a.shape[0], a.shape[1], _ptr(gx), _ptr(gy)))
    return gx, gy


def cuda_sobel(blur, ctx: Optional[Context] = None) -> Tuple[np.ndarray, np.ndarray]:
    a = _img(blur, np.int16)
    mag, ang = np.empty(a.shape, np.int16), np.empty(a.shape, np.int16)
    check(load().b200_sobel(_h(ctx), _ptr(a), a.shape[0], a.shape[1], _ptr(mag), _ptr(ang)))
    return mag, ang


def cuda_nonmaixmal_suppression(magnitude, angle, ctx: Optional[Context] = None) -> np.ndarray:
    m, a = _img(magnitude, np.int16), _img(angle, np.int16)
    if m.shape != a.shape:
        raise ValueError("magnitude and angle must have the same shape")
    out = np.empty(m.shape, np.int16)
    check(load().b200_nonmaximal(_h(ctx), _ptr(m), _ptr(a), m.shape[0], m.shape[1], _ptr(out)))
    return out


def cuda_hysteresis(nms, min_val: int, max_val: int, ctx: Optional[Context] = None) -> np.ndarray:
    """hysteresis (src/utils.cpp:322-342) on the GPU; returns the 0/255 map (the reference works in place)."""
    a = _img(nms, np.int16).copy()
    check(load().b200_hysteresis(_h(ctx), _ptr(a), a.shape[0], a.shape[1], int(min_val), int(max_val)))
    return a


def cuda_canny(img, sigma: float, min_val: int, max_val: int, steps: bool = False, ctx: Optional[Context] = None):
    """cuda_canny (src/cuda.cu:392-450).  Returns the int16 0/255 edge map; with steps=True returns
    (blur, magnitude, angle, nms, edges) — the planes the reference displays after each stage."""
    a = _img(img, np.uint8)
    h, w = a.shape
    edges = np.empty((h, w), np.int16)
    if not steps:
        check(load().b200_canny(_h(ctx), _ptr(a), C.c_float(sigma), int(min_val), int(max_val), h, w, _ptr(edges)))
        return edges
    blur, mag, ang, nms = (np.empty((h, w), np.int16) for _ in range(4))
    check(load().b200_canny_steps(_h(ctx), _ptr(a), C.c_float(sigma), int(min_val), int(max_val), h, w, _ptr(blur),
                                  _ptr(mag), _ptr(ang), _ptr(nms), _ptr(edges)))
    return blur, mag, ang, nms, edges


def cuda_canny_bgr(frame, sigma: float, min_val: int, max_val: int, return_gray: bool = False, ctx: Optional[Context] = None):
    """One interleaved B,G,R frame (h, w, 3) as cv2 / cv::Mat hold it: cvtColor(BGR2GRAY) + cuda_canny on the GPU — the
    reference's per-frame work, src/main.cpp:113,128.  Returns the int16 0/255 map (and the uint8 gray plane when asked)."""
    a = np.ascontiguousarray(frame, dtype=np.uint8)
    if a.ndim != 3 or a.shape[2] != 3:
        raise ValueError("expected a (height, width, 3) BGR frame")
    h, w = a.shape[:2]
    edges = np.empty((h, w), np.int16)
    gray = np.empty((h, w), np.uint8) if return_gray else None
    check(load().b200_canny_bgr(_h(ctx), _ptr(a), C.c_float(sigma), int(min_val), int(max_val), h, w,
                                _ptr(gray) if return_gray else None, _ptr(edges)))
    return (edges, gray) if return_gray else edges


# ---------------------------------------------------------------------------------------------------
# batched
# ---------------------------------------------------------------------------------------------------
def canny_batch_host(frames, sigma: float, min_val: int, max_val: int, out: Optional[np.ndarray] = None,
                     ctx: Optional[Context] = None) -> np.ndarray:
    """(n, h, w) uint8 host frames -> (n, h, w) uint8 0/255, copies pipelined against the kernels."""
    a = np.ascontiguousarray(frames, dtype=np.uint8)
    if a.ndim != 3:
        raise ValueError("expected (n_frames, height, width)")
    n, h, w = a.shape
    if out is None:
        out = np.empty_like(a)
    check(load().b200_canny_batch_host(_h(ctx), _ptr(a), n, h, w, C.c_float(sigma), int(min_val), int(max_val), _ptr(out)))
    return out


def canny_batch_device_ptr(ctx: Context, d_frames: int, n: int, h: int, w: int, sigma: float, min_val: int,
                           max_val: int, d_edges: int) -> None:
    """Raw device pointers (e.g. torch tensor.data_ptr()); asynchronous on the context's stream."""
    check(load().b200_canny_batch_device(_h(ctx), C.c_void_p(d_frames), n, h, w, C.c_float(sigma), int(min_val),
                                         int(max_val), C.c_void_p(d_edges)))


def canny_batch_device_bgr_ptr(ctx: Context, d_bgr: int, n: int, h: int, w: int, sigma: float, min_val: int,
                               max_val: int, d_edges: int) -> None:
    """Device-resident interleaved B,G,R frames (n, h, w, 3) -> u8 edge maps; cvtColor(BGR2GRAY) (src/main.cpp:113) runs inside
    the front kernel's staging when the shape allows (b200_canny_batch_device_bgr).  Asynchronous on the context's stream."""
    check(load().b200_canny_batch_device_bgr(_h(ctx), C.c_void_p(d_bgr), n, h, w, C.c_float(sigma), int(min_val),
                                             int(max_val), C.c_void_p(d_edges)))


def canny_batch_device_strided_ptr(ctx: Optional[Context], d_frames: int, in_row_pitch: int, in_frame_stride: int, n: int, h: int,
                                   w: int, sigma: float, min_val: int, max_val: int, d_edges: int, out_row_pitch: int,
                                   out_frame_stride: int) -> None:
    """Raw device pointers with byte strides (b200_canny_batch_device_strided): pixel (f, y, x) is read at
    d_frames + f*in_frame_stride + y*in_row_pitch + x and written at d_edges + f*out_frame_stride + y*out_row_pitch + x; no other
    byte of the output is touched.  Asynchronous on the context's stream."""
    check(load().b200_canny_batch_device_strided(_h(ctx), C.c_void_p(d_frames), int(in_row_pitch), int(in_frame_stride), n, h, w,
                                                 C.c_float(sigma), int(min_val), int(max_val), C.c_void_p(d_edges),
                                                 int(out_row_pitch), int(out_frame_stride)))


def canny_batch_device_bgr_strided_ptr(ctx: Optional[Context], d_bgr: int, in_row_pitch: int, in_frame_stride: int, n: int, h: int,
                                       w: int, sigma: float, min_val: int, max_val: int, d_edges: int, out_row_pitch: int,
                                       out_frame_stride: int) -> None:
    """Interleaved B,G,R frames with byte strides (b200_canny_batch_device_bgr_strided): pixel (f, y, x) is the 3 bytes at
    d_bgr + f*in_frame_stride + y*in_row_pitch + 3*x.  Asynchronous on the context's stream."""
    check(load().b200_canny_batch_device_bgr_strided(_h(ctx), C.c_void_p(d_bgr), int(in_row_pitch), int(in_frame_stride), n, h, w,
                                                     C.c_float(sigma), int(min_val), int(max_val), C.c_void_p(d_edges),
                                                     int(out_row_pitch), int(out_frame_stride)))


def cv_canny_device_strided_ptr(ctx: Optional[Context], d_in: int, in_row_pitch: int, in_frame_stride: int, n: int, h: int, w: int,
                                channels: int, threshold1: float, threshold2: float, l2_gradient: bool, d_edges: int,
                                out_row_pitch: int, out_frame_stride: int, aperture_size: int = 3) -> None:
    """cv2.Canny(frame, threshold1, threshold2, apertureSize=aperture_size, L2gradient=l2_gradient) of every frame, bit for bit
    (b200_cv_canny_aperture_device_strided; aperture_size 3, 5 or 7): 1 or 3 interleaved channels, pixel (f, y, x) read at
    d_in + f*in_frame_stride + y*in_row_pitch + channels*x, its 0 / 255 result written at d_edges + f*out_frame_stride +
    y*out_row_pitch + x.  Asynchronous on the context's stream."""
    check(load().b200_cv_canny_aperture_device_strided(_h(ctx), C.c_void_p(d_in), int(in_row_pitch), int(in_frame_stride), n, h, w,
                                                       int(channels), C.c_double(threshold1), C.c_double(threshold2),
                                                       int(aperture_size), int(bool(l2_gradient)), C.c_void_p(d_edges),
                                                       int(out_row_pitch), int(out_frame_stride)))


def frame_list(descs) -> C.Array:
    """(in_ptr, in_pitch, out_ptr, out_pitch, h, w) tuples -> the ctypes array of b200_frame that b200_canny_frames_device takes."""
    descs = list(descs)
    arr = (_lib.Frame * max(1, len(descs)))()
    for i, (in_ptr, in_pitch, out_ptr, out_pitch, h, w) in enumerate(descs):
        arr[i] = _lib.Frame(in_ptr, int(in_pitch), out_ptr, int(out_pitch), int(h), int(w))
    return arr


def canny_frames_device_ptr(ctx: Optional[Context], descs, sigma: float, min_val: int, max_val: int, bgr: bool = False) -> None:
    """Frames of different sizes in one call (b200_canny_frames_device[_bgr]).  descs: a sequence of (in_ptr, in_pitch, out_ptr,
    out_pitch, h, w) with device pointers and byte pitches: pixel (y, x) of a frame is read at in_ptr + y*in_pitch + x (3 bytes at
    + 3*x for B,G,R) and written at out_ptr + y*out_pitch + x.  Asynchronous on the context's stream."""
    descs = list(descs)
    fn = load().b200_canny_frames_device_bgr if bgr else load().b200_canny_frames_device
    check(fn(_h(ctx), frame_list(descs), len(descs), C.c_float(sigma), int(min_val), int(max_val)))


def cv_canny_frames_device_ptr(ctx: Optional[Context], descs, channels: int, threshold1: float, threshold2: float,
                               l2_gradient: bool, aperture_size: int = 3) -> None:
    """cv2.Canny(frame, threshold1, threshold2, apertureSize=aperture_size, L2gradient=l2_gradient) of frames of different sizes in
    one call, bit for bit (b200_cv_canny_aperture_frames_device; aperture_size 3, 5 or 7).  descs as canny_frames_device_ptr: pixel
    (y, x) of a frame is the `channels` bytes (1 or 3 interleaved) at in_ptr + y*in_pitch + channels*x, its 0 / 255 result written
    at out_ptr + y*out_pitch + x; frames from 1 x 1.  Asynchronous on the context's stream."""
    descs = list(descs)
    check(load().b200_cv_canny_aperture_frames_device(_h(ctx), frame_list(descs), len(descs), int(channels), C.c_double(threshold1),
                                                      C.c_double(threshold2), int(aperture_size), int(bool(l2_gradient))))


def synth_host(n: int, h: int, w: int, kind: int = 0, seed: int = 1234, first_frame: int = 0) -> np.ndarray:
    out = np.empty((n, h, w), np.uint8)
    check(load().b200_synth_host(_ptr(out), n, h, w, kind, C.c_uint64(seed), first_frame))
    return out


def synth_rows_host(row0: int, rows: int, w: int, kind: int = 0, seed: int = 1234, frame: int = 0) -> np.ndarray:
    out = np.empty((rows, w), np.uint8)
    check(load().b200_synth_rows_host(_ptr(out), row0, rows, w, kind, C.c_uint64(seed), frame))
    return out
