"""torch front end of the device batch path: CUDA uint8 tensors in, uint8 0/255 tensors out.

Any view whose rows are contiguous goes straight to the kernels with its strides — a crop `x[:, y0:y1, x0:x1]`, one channel of an
`(N, C, H, W)` tensor, frames padded for alignment — through b200_canny_batch_device_strided; nothing is copied.  Layouts the
kernels cannot address (rows that are not unit-stride, frames that overlap, broadcast frames) raise ValueError rather than being
copied behind the caller's back.  canny_list / canny_bgr_list take a list of frames of different sizes in one call
(b200_canny_frames_device).  cv_canny / cv_canny_color compute cv2.Canny's maps instead of the reference's
(b200_cv_canny_aperture_device_strided; apertureSize 3, 5 or 7), from the same kinds of views; cv_canny_list / cv_canny_color_list
do so for lists of frames of different sizes (b200_cv_canny_aperture_frames_device).

Work is issued on torch.cuda.current_stream(frames.device): the context is pointed at that stream on every call, so results are
ordered with the caller's other torch work like any torch op.  When consecutive calls come from different streams, the later
stream first waits for the earlier call (b200_ctx_set_stream), because calls on one context share its workspace.  torch is imported inside the functions, as in sharded.py.
"""
from __future__ import annotations

import threading
from typing import Dict, Optional, Tuple

from .api import (Context, canny_batch_device_bgr_strided_ptr, canny_batch_device_strided_ptr, canny_frames_device_ptr,
                  cv_canny_device_strided_ptr, cv_canny_frames_device_ptr)

_contexts: Dict[int, Context] = {}
_contexts_lock = threading.Lock()
_call_lock = threading.Lock()   # a context's stream is state: pointing it at a stream and issuing the call happen together

_CUDA_STREAM_LEGACY = 0x1   # cudaStreamLegacy (driver_types.h)
_CONTIGUOUS_HINT = "pass a view whose rows are contiguous (e.g. call .contiguous() first)"


def frame_layout(t, bgr: bool = False, min_side: int = 2) -> Tuple[int, int, int, int, int]:
    """(n_frames, height, width, row pitch, frame stride) of a uint8 tensor as the strided C calls take them, strides in bytes.

    Gray: (H, W) or (N, H, W).  BGR: (H, W, 3) or (N, H, W, 3).  Raises ValueError for a layout the kernels cannot address, or for
    frames smaller than min_side x min_side (2 for the reference's semantics, 1 for the OpenCV-compatible calls)."""
    import torch

    if not isinstance(t, torch.Tensor):
        raise TypeError(f"expected a torch.Tensor, got {type(t).__name__}")
    if t.dtype != torch.uint8:
        raise ValueError(f"expected a uint8 tensor, got {t.dtype}")
    shape, stride = tuple(t.shape), tuple(t.stride())
    if bgr:
        if t.dim() not in (3, 4) or shape[-1] != 3:
            raise ValueError(f"expected (H, W, 3) or (N, H, W, 3) B,G,R frames, got shape {shape}")
        if stride[-1] != 1 or stride[-2] != 3:
            raise ValueError(f"B,G,R pixels must be 3 contiguous bytes (strides (..., 3, 1), got {stride}); {_CONTIGUOUS_HINT}")
        shape, stride = shape[:-1], stride[:-1]
        row_bytes = 3 * shape[-1]
    else:
        if t.dim() not in (2, 3):
            raise ValueError(f"expected (H, W) or (N, H, W) gray frames, got shape {shape}")
        if stride[-1] != 1:
            raise ValueError(f"rows must be contiguous (last stride 1, got {stride}); {_CONTIGUOUS_HINT}")
        row_bytes = shape[-1]
    h, w = shape[-2], shape[-1]
    pitch = stride[-2]
    n = shape[0] if len(shape) == 3 else 1
    if h < min_side or w < min_side:
        raise ValueError(f"frames must be at least {min_side} x {min_side} pixels (got {h} x {w})")
    if n < 1:
        raise ValueError("no frames")
    if pitch < row_bytes:
        raise ValueError(f"rows overlap (row stride {pitch} < {row_bytes} bytes per row); {_CONTIGUOUS_HINT}")
    frame_bytes = (h - 1) * pitch + row_bytes
    frame_stride = stride[0] if len(shape) == 3 else h * pitch
    if n > 1 and frame_stride < frame_bytes:
        raise ValueError(f"frames overlap or are broadcast (frame stride {frame_stride} < {frame_bytes} bytes per frame); "
                         f"{_CONTIGUOUS_HINT}")
    if n == 1:
        frame_stride = h * pitch
    return n, h, w, pitch, frame_stride


def _context(device_index: int) -> Context:
    with _contexts_lock:
        ctx = _contexts.get(device_index)
        if ctx is None:
            ctx = _contexts[device_index] = Context(device_index)
        return ctx


def _run(frames, sigma: float, min_val: int, max_val: int, out, ctx: Optional[Context], bgr: bool, cv_l2=None, aperture: int = 3):
    """cv_l2 None: the reference's Canny (sigma, min_val, max_val); False / True: cv2.Canny with L1 / L2 magnitude and Sobel
    aperture `aperture`, min_val and max_val being threshold1 and threshold2."""
    import torch

    min_side = 2 if cv_l2 is None else 1
    n, h, w, in_pitch, in_fs = frame_layout(frames, bgr, min_side)
    out_shape = tuple(frames.shape[:-1]) if bgr else tuple(frames.shape)
    if not frames.is_cuda:
        raise ValueError(f"frames must be a CUDA tensor (got device {frames.device})")
    if out is None:
        out = torch.empty(out_shape, dtype=torch.uint8, device=frames.device)
    else:
        if tuple(out.shape) != out_shape:
            raise ValueError(f"out has shape {tuple(out.shape)}, expected {out_shape}")
        if out.device != frames.device:
            raise ValueError(f"out is on {out.device}, frames on {frames.device}")
    _, _, _, out_pitch, out_fs = frame_layout(out, False, min_side)
    dev = frames.device.index if frames.device.index is not None else torch.cuda.current_device()
    if ctx is None:
        ctx = _context(dev)
    elif ctx.device != dev:
        raise ValueError(f"context is on cuda:{ctx.device}, frames on cuda:{dev}")
    with _call_lock, torch.cuda.device(dev):
        # torch's default stream has the handle 0, which the library reads as "the context's own stream": name the legacy default
        # stream (cudaStreamLegacy) instead, so the work is ordered with the caller's
        ctx.set_stream(torch.cuda.current_stream(dev).cuda_stream or _CUDA_STREAM_LEGACY)
        if cv_l2 is not None:
            cv_canny_device_strided_ptr(ctx, frames.data_ptr(), in_pitch, in_fs, n, h, w, 3 if bgr else 1, min_val, max_val, cv_l2,
                                        out.data_ptr(), out_pitch, out_fs, aperture)
        else:
            call = canny_batch_device_bgr_strided_ptr if bgr else canny_batch_device_strided_ptr
            call(ctx, frames.data_ptr(), in_pitch, in_fs, n, h, w, sigma, min_val, max_val, out.data_ptr(), out_pitch, out_fs)
    return out


def canny(frames, sigma: float, min_val: int, max_val: int, *, out=None, ctx: Optional[Context] = None):
    """Canny edge maps of gray frames: a CUDA uint8 tensor of shape (H, W) or (N, H, W), any strides with contiguous rows.

    Returns a uint8 tensor of the same shape holding 0 / 255 (`out` when given: it may be a strided view, only its elements are
    written).  Asynchronous on torch.cuda.current_stream(frames.device); ctx defaults to one cached Context per device."""
    return _run(frames, sigma, min_val, max_val, out, ctx, bgr=False)


def canny_bgr(frames, sigma: float, min_val: int, max_val: int, *, out=None, ctx: Optional[Context] = None):
    """canny() for interleaved B,G,R frames (cv2 / cv::Mat layout): (H, W, 3) or (N, H, W, 3), each pixel's 3 bytes contiguous,
    rows and frames with any stride.  The gray conversion is OpenCV's COLOR_BGR2GRAY, bit for bit.  Returns (H, W) or (N, H, W)."""
    return _run(frames, sigma, min_val, max_val, out, ctx, bgr=True)


def cv_canny(frames, threshold1: float, threshold2: float, *, apertureSize: int = 3, L2gradient: bool = False, out=None,
             ctx: Optional[Context] = None):
    """cv2.Canny(frame, threshold1, threshold2, apertureSize=apertureSize, L2gradient=L2gradient) of gray frames, bit for bit: a
    CUDA uint8 tensor of shape (H, W) or (N, H, W), any strides with contiguous rows, frames of at least 1 x 1.

    No blur, Sobel of apertureSize 3, 5 or 7 with replicated borders (7: derivatives and thresholds scaled by 1/16, as cv2 does),
    L1 (or L2) magnitude, OpenCV's direction test and non-maximum suppression, `> low` / `> high` thresholds (swapped when
    threshold1 > threshold2), plain 8-connected hysteresis.  Any other apertureSize raises CannyB200Error, as cv2 rejects it.
    Returns a uint8 tensor of the same shape holding 0 / 255 (`out` when given, which may be a strided view).  Asynchronous on
    torch.cuda.current_stream(frames.device); ctx defaults to one cached Context per device."""
    return _run(frames, 0.0, float(threshold1), float(threshold2), out, ctx, bgr=False, cv_l2=bool(L2gradient),
                aperture=int(apertureSize))


def cv_canny_color(frames, threshold1: float, threshold2: float, *, apertureSize: int = 3, L2gradient: bool = False, out=None,
                   ctx: Optional[Context] = None):
    """cv2.Canny of 3-channel frames, bit for bit: (H, W, 3) or (N, H, W, 3), each pixel's 3 bytes contiguous, rows and frames with
    any stride; apertureSize 3, 5 or 7.  As cv2.Canny on a 3-channel image: the gradient of every channel, per pixel the channel
    of largest magnitude.  The channel order does not matter (B,G,R or R,G,B give the same map except where two channels tie,
    when the first wins).  Returns (H, W) or (N, H, W)."""
    return _run(frames, 0.0, float(threshold1), float(threshold2), out, ctx, bgr=True, cv_l2=bool(L2gradient),
                aperture=int(apertureSize))


def _run_list(frames, sigma: float, min_val: int, max_val: int, out, ctx: Optional[Context], bgr: bool, cv_l2=None,
              aperture: int = 3):
    """cv_l2 and aperture as _run: cv_l2 None for the reference's Canny, False / True for cv2.Canny with L1 / L2 magnitude."""
    import torch

    min_side = 2 if cv_l2 is None else 1
    frames = list(frames)
    if not frames:
        raise ValueError("empty frame list")
    single = 3 if bgr else 2   # one frame per element: (H, W) gray, (H, W, 3) B,G,R
    descs = []
    for i, f in enumerate(frames):
        if isinstance(f, torch.Tensor) and f.dim() != single:
            raise ValueError(f"frame {i}: expected one {'(H, W, 3) B,G,R' if bgr else '(H, W) gray'} frame, got shape {tuple(f.shape)}")
        _, h, w, pitch, _ = frame_layout(f, bgr, min_side)
        descs.append([f.data_ptr(), pitch, 0, 0, h, w])
    if out is not None:
        out = list(out)
        if len(out) != len(frames):
            raise ValueError(f"out has {len(out)} tensors for {len(frames)} frames")
        for i, (o, d) in enumerate(zip(out, descs)):
            if not isinstance(o, torch.Tensor) or tuple(o.shape) != (d[4], d[5]):
                raise ValueError(f"out[{i}] has shape {tuple(getattr(o, 'shape', ()))}, expected {(d[4], d[5])}")
    device = frames[0].device
    for i, t in enumerate(frames + (out or [])):
        name = f"frame {i}" if i < len(frames) else f"out[{i - len(frames)}]"
        if not t.is_cuda:
            raise ValueError(f"{name} must be a CUDA tensor (got device {t.device})")
        if t.device != device:
            raise ValueError(f"{name} is on {t.device}, frame 0 on {device}: all tensors must be on one device")
    if out is None:
        out = [torch.empty((d[4], d[5]), dtype=torch.uint8, device=device) for d in descs]
    for d, o in zip(descs, out):
        _, _, _, d[3], _ = frame_layout(o, False, min_side)
        d[2] = o.data_ptr()
    dev = device.index if device.index is not None else torch.cuda.current_device()
    if ctx is None:
        ctx = _context(dev)
    elif ctx.device != dev:
        raise ValueError(f"context is on cuda:{ctx.device}, frames on cuda:{dev}")
    with _call_lock, torch.cuda.device(dev):
        ctx.set_stream(torch.cuda.current_stream(dev).cuda_stream or _CUDA_STREAM_LEGACY)
        if cv_l2 is not None:
            cv_canny_frames_device_ptr(ctx, descs, 3 if bgr else 1, min_val, max_val, cv_l2, aperture)
        else:
            canny_frames_device_ptr(ctx, descs, sigma, min_val, max_val, bgr=bgr)
    return out


def canny_list(frames, sigma: float, min_val: int, max_val: int, *, out=None, ctx: Optional[Context] = None):
    """Canny edge maps of a list of gray frames of different sizes, in one call (b200_canny_frames_device): each element a CUDA
    uint8 (H, W) view whose rows are contiguous, any row pitch.  Returns a list of uint8 (H, W) tensors holding 0 / 255 (`out` when
    given: a list of views of the same shapes, e.g. regions of one mosaic; only their elements are written).  Every map equals
    canny() of that frame alone.  Asynchronous on torch.cuda.current_stream(device); ctx defaults to the cached Context."""
    return _run_list(frames, sigma, min_val, max_val, out, ctx, bgr=False)


def canny_bgr_list(frames, sigma: float, min_val: int, max_val: int, *, out=None, ctx: Optional[Context] = None):
    """canny_list() for interleaved B,G,R frames: each element an (H, W, 3) view with each pixel's 3 bytes contiguous.  The gray
    conversion is OpenCV's COLOR_BGR2GRAY, bit for bit.  Returns a list of (H, W) maps."""
    return _run_list(frames, sigma, min_val, max_val, out, ctx, bgr=True)


def cv_canny_list(frames, threshold1: float, threshold2: float, *, apertureSize: int = 3, L2gradient: bool = False, out=None,
                  ctx: Optional[Context] = None):
    """cv2.Canny(frame, threshold1, threshold2, apertureSize=apertureSize, L2gradient=L2gradient) of a list of gray frames of
    different sizes, in one call (b200_cv_canny_aperture_frames_device; apertureSize 3, 5 or 7, anything else raises
    CannyB200Error): each element a CUDA uint8 (H, W) view whose rows are contiguous, any row pitch, at least 1 x 1.  Returns a list of uint8 (H, W) tensors holding 0 / 255 (`out` when given: a list of views of the same shapes, e.g.
    tiles of one mosaic; only their elements are written).  Every map equals cv_canny() of that frame alone.  Asynchronous on
    torch.cuda.current_stream(device); ctx defaults to the cached Context."""
    return _run_list(frames, 0.0, float(threshold1), float(threshold2), out, ctx, bgr=False, cv_l2=bool(L2gradient),
                     aperture=int(apertureSize))


def cv_canny_color_list(frames, threshold1: float, threshold2: float, *, apertureSize: int = 3, L2gradient: bool = False,
                        out=None, ctx: Optional[Context] = None):
    """cv_canny_list() for 3-channel frames: each element an (H, W, 3) view with each pixel's 3 bytes contiguous; apertureSize 3,
    5 or 7.  Every map equals cv_canny_color() of that frame alone.  Returns a list of (H, W) maps."""
    return _run_list(frames, 0.0, float(threshold1), float(threshold2), out, ctx, bgr=True, cv_l2=bool(L2gradient),
                     aperture=int(apertureSize))
