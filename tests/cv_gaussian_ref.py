"""TEST INFRASTRUCTURE ONLY: cv::GaussianBlur (OpenCV 4.x, 8-bit input, default border) restated in numpy, bit for bit.

The specification of the blur of b200_cv_gaussian_canny_device_strided and b200_cv_gaussian_canny_frames_device; Canny on the
blurred frame is tests/cv_canny_aperture_ref.py.  Checked against cv2.GaussianBlur by tests/test_cv_gaussian_cpu.py wherever cv2 is
importable.

    Arguments: sigmaY <= 0 means sigmaX; a ksize side <= 0 is derived from its sigma when that is > 0, cvRound(sigma*3*2 + 1) | 1
    (half to even); both sides must then be odd and positive; negative sigmas count as 0.
    Taps per axis: getGaussianKernelBitExact (OpenCV's fixed tables for sigma 0 and n = 1, 3, 5, 7; else exp(-x^2 / (8 s^2)) at
    x = 1-n, 3-n, ... normalised, s = sigma or 0.15 n + 0.35 by one fma), then each half rounded to 1/256 with the error carried
    from tap to tap (half to even) and the centre tap making the sum 256.
    Blur: (sum_i sum_j fy[i] fx[j] I(r(y+i-ry), r(x+j-rx)) + 2^15) >> 16, r reflect-101 with period 2(len-1), a 1-pixel side
    always index 0.  Every sum is an exact integer.

cv2 as a reference runs on one thread (cv2_gaussian_blur): cv2 4.13 (IPP build) with several threads returns, now and then, a
different result for the same (5, 5) sigma-0 call (a few pixels off by up to 10, and the next identical call gives the other
result); on one thread its result is the same every time and equals this restatement.
"""
from __future__ import annotations

import contextlib
import math
from fractions import Fraction

import numpy as np

MAX_KSIZE = 31
SMALL = {1: [1.0], 3: [0.25, 0.5, 0.25], 5: [1 / 16, 4 / 16, 6 / 16, 4 / 16, 1 / 16],
         7: [1 / 32, 3.5 / 32, 7 / 32, 9 / 32, 7 / 32, 3.5 / 32, 1 / 32]}


class GaussArgError(ValueError):
    """Arguments cv2.GaussianBlur rejects (status: the library's code, 1 = invalid argument) or this build does not take (4)."""

    def __init__(self, status: int, msg: str):
        super().__init__(msg)
        self.status = status


def cv_round(v: float) -> int:
    """cvRound: nearest integer, half to even."""
    return int(round(v))


def _fma(a: float, b: float, c: float) -> float:
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def resolve(ksize, sigma_x: float, sigma_y: float = 0.0):
    """((kw, kh), sx, sy) as cv2.GaussianBlur resolves its arguments; GaussArgError for what the library refuses."""
    kw, kh = (ksize, ksize) if isinstance(ksize, int) else ksize
    if not (math.isfinite(sigma_x) and math.isfinite(sigma_y)):
        raise GaussArgError(1, "sigma must be finite")
    if sigma_y <= 0:
        sigma_y = sigma_x
    if kw <= 0 and sigma_x > 0:
        kw = cv_round(sigma_x * 3 * 2 + 1) | 1
    if kh <= 0 and sigma_y > 0:
        kh = cv_round(sigma_y * 3 * 2 + 1) | 1
    if kw <= 0 or kh <= 0 or kw % 2 == 0 or kh % 2 == 0:
        raise GaussArgError(1, f"ksize ({kw}, {kh}) must be odd and positive")
    if kw > MAX_KSIZE or kh > MAX_KSIZE:
        raise GaussArgError(4, f"ksize ({kw}, {kh}) above {MAX_KSIZE}")
    return (kw, kh), max(sigma_x, 0.0), max(sigma_y, 0.0)


def kernel_bitexact(n: int, sigma: float):
    """getGaussianKernelBitExact's double taps for n (odd) and sigma >= 0."""
    if sigma <= 0 and n in SMALL:
        return list(SMALL[n])
    s = sigma if sigma > 0 else _fma(float(n), 0.15, 0.35)
    c = -0.125 / (s * s)
    h = (n - 1) // 2
    t = []
    total = 0.0
    for i in range(h):
        x = 1 - n + 2 * i
        t.append(math.exp(float(x * x) * c))
        total += t[-1]
    total = total * 2.0 + 1.0
    m = 1.0 / total
    k = [0.0] * n
    for i in range(h):
        k[i] = k[n - 1 - i] = t[i] * m
    k[h] = 1.0 * m
    return k


def fixed_taps(n: int, sigma: float) -> np.ndarray:
    """The 8.8 fixed-point taps (int64, summing to 256) of n and sigma >= 0, as b200_cv_gaussian_kernel returns them."""
    k = kernel_bitexact(n, sigma)
    out = [0] * n
    err = 0.0
    acc = 0
    for i in range(n // 2):
        a = k[i] * 256.0 + err
        v = cv_round(a)
        err = a - float(v)
        out[i] = out[n - 1 - i] = v
        acc += v
    out[n // 2] = 256 - 2 * acc
    return np.array(out, np.int64)


def kernel(ksize: int, sigma: float):
    """(resolved size, taps) of one axis, as b200_cv_gaussian_kernel(ksize, sigma)."""
    (n, _), s, _ = resolve((ksize, ksize), sigma, sigma)
    return n, fixed_taps(n, s)


def reflect101(n: int, idx: np.ndarray) -> np.ndarray:
    """BORDER_REFLECT_101 indices into 0 .. n-1, repeated with period 2(n-1); a 1-pixel side always maps to 0."""
    idx = np.asarray(idx, np.int64)
    if n == 1:
        return np.zeros_like(idx)
    per = 2 * (n - 1)
    idx = np.mod(idx, per)
    return np.where(idx < n, idx, per - idx)


def gaussian_blur(img, ksize, sigma_x: float, sigma_y: float = 0.0) -> np.ndarray:
    """cv2.GaussianBlur(img, ksize, sigma_x, sigmaY=sigma_y) of an (H, W) or (H, W, C) uint8 image, bit for bit; ksize an int
    (square) or (width, height)."""
    (kw, kh), sx, sy = resolve(ksize, sigma_x, sigma_y)
    fx, fy = fixed_taps(kw, sx), fixed_taps(kh, sy)
    a = np.asarray(img).astype(np.int64)
    gray = a.ndim == 2
    if gray:
        a = a[..., None]
    H, W, _ = a.shape
    rx, ry = kw // 2, kh // 2
    p = a[reflect101(H, np.arange(-ry, H + ry))][:, reflect101(W, np.arange(-rx, W + rx))]
    h = sum(fx[j] * p[:, j:j + W] for j in range(kw))
    v = sum(fy[i] * h[i:i + H] for i in range(kh))
    out = ((v + 32768) >> 16).astype(np.uint8)
    return out[..., 0] if gray else out


@contextlib.contextmanager
def cv2_one_thread(cv2):
    """cv2 on one thread for the duration (its multi-threaded (5, 5) sigma-0 blur is not deterministic; see the module notes)."""
    n = cv2.getNumThreads()
    cv2.setNumThreads(1)
    try:
        yield
    finally:
        cv2.setNumThreads(n)


def cv2_gaussian_blur(cv2, img, ksize, sigma_x: float, sigma_y: float = 0.0) -> np.ndarray:
    """cv2.GaussianBlur(img, ksize, sigma_x, sigmaY=sigma_y), computed on one thread."""
    with cv2_one_thread(cv2):
        return cv2.GaussianBlur(np.ascontiguousarray(img), ksize, sigma_x, sigmaY=sigma_y)


def cv_gaussian_canny(img, ksize, sigma_x: float, sigma_y: float, lo: float, hi: float, l2: bool = False, aperture: int = 3):
    """cv2.Canny(cv2.GaussianBlur(img, ksize, sigma_x, sigmaY=sigma_y), lo, hi, apertureSize=aperture, L2gradient=l2)."""
    from cv_canny_aperture_ref import cv_canny

    return cv_canny(gaussian_blur(img, ksize, sigma_x, sigma_y), lo, hi, l2, aperture)
