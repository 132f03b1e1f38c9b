"""TEST INFRASTRUCTURE ONLY: cv::Canny (OpenCV 4.x) with apertureSize 3, 5 or 7, restated in numpy, bit for bit.

The specification of b200_cv_canny_aperture_device_strided and b200_cv_canny_aperture_frames_device.  Aperture 3 is
oracle/cv_canny.py itself; 5 and 7 follow the same rules with cv::getDerivKernels' wider taps.  Checked against cv2.Canny by
tests/test_cv_aperture_cpu.py wherever cv2 is importable.

    Sobel K x K, separable, BORDER_REPLICATE for both derivatives: dx is the derivative taps across columns and the smoothing taps
    down rows, dy the transpose.
      K = 5: smoothing 1 4 6 4 1, derivative -1 -2 0 2 1; exact integers (|dx|, |dy| <= 12240).
      K = 7: smoothing 1 6 15 20 15 6 1, derivative -1 -4 -5 0 5 4 1; both derivatives are the exact sum S scaled by 1/16 and
             rounded half to even (cvRound): floor(S / 16), plus 1 when the remainder is above 8, or 8 with an odd quotient.
             Both thresholds are divided by 16 first, before the swap, the L2 clamp, the squaring and the floor.
    Then as at aperture 3: per pixel the channel of largest magnitude (the first on ties), |dx|+|dy| (L1) or dx^2+dy^2 (L2, against
    squared thresholds); direction by the fixed-point tan(22.5 deg) test; non-maximum suppression with `>` on one side and `>=` on
    the other (both `>` on diagonals); `> low` candidates, `> high` seeds; plain 8-connected hysteresis.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage

from oracle import cv_canny as cv3

APERTURES = (3, 5, 7)
SMOOTH = {3: (1, 2, 1), 5: (1, 4, 6, 4, 1), 7: (1, 6, 15, 20, 15, 6, 1)}
DERIV = {3: (-1, 0, 1), 5: (-1, -2, 0, 2, 1), 7: (-1, -4, -5, 0, 5, 4, 1)}


def _check(aperture):
    if aperture not in APERTURES:
        raise ValueError(f"aperture must be 3, 5 or 7 (got {aperture})")


def cv_thresholds(lo: float, hi: float, l2: bool = False, aperture: int = 3):
    """(low, high) as integers in magnitude space, as cv::Canny derives them: divided by 16 for aperture 7, then swapped when
    low > high, clamped and squared for L2, floored."""
    _check(aperture)
    if aperture == 7:
        lo, hi = lo / 16, hi / 16
    return cv3.cv_thresholds(lo, hi, l2)


def sobel_sums(img, aperture: int):
    """The exact integer K x K Sobel sums (dx, dy) of every pixel and channel, (H, W, C) int64 each, before any scaling."""
    _check(aperture)
    img = np.asarray(img).astype(np.int64)
    if img.ndim == 2:
        img = img[..., None]
    H, W, _ = img.shape
    r = aperture // 2
    p = np.pad(img, ((r, r), (r, r), (0, 0)), mode="edge")                  # BORDER_REPLICATE
    s, d = SMOOTH[aperture], DERIV[aperture]
    across_d = sum(d[t] * p[:, t:t + W] for t in range(aperture))            # per padded row: derivative taps across columns
    across_s = sum(s[t] * p[:, t:t + W] for t in range(aperture))            # ... and smoothing taps
    dx = sum(s[i] * across_d[i:i + H] for i in range(aperture))
    dy = sum(d[i] * across_s[i:i + H] for i in range(aperture))
    return dx, dy


def cv_round16(s):
    """cvRound(s / 16) of integers s, in integers: half to even."""
    q, r = np.floor_divide(s, 16), np.mod(s, 16)
    return q + ((r > 8) | ((r == 8) & (q % 2 == 1)))


def cv_gradients(img, aperture: int):
    """(dx, dy) as cv::Canny computes them: the Sobel sums, scaled by 1/16 with cvRound for aperture 7."""
    dx, dy = sobel_sums(img, aperture)
    if aperture == 7:
        dx, dy = cv_round16(dx), cv_round16(dy)
    return dx, dy


def canny_from_gradients(dx, dy, lo: int, hi: int, l2: bool = False):
    """The 0 / 255 map from per-channel gradients (H, W, C) and integer thresholds in magnitude space (cv_thresholds)."""
    dx, dy = np.asarray(dx, np.int64), np.asarray(dy, np.int64)
    H, W, _ = dx.shape
    n = dx * dx + dy * dy if l2 else np.abs(dx) + np.abs(dy)
    k = np.argmax(n, axis=2)                                                 # first channel of maximal magnitude
    ii, jj = np.indices((H, W))
    m, gx, gy = n[ii, jj, k], dx[ii, jj, k], dy[ii, jj, k]
    M = np.pad(m, 1)                                                         # magnitude outside the image is 0

    def c(di, dj):
        return M[1 + di:1 + di + H, 1 + dj:1 + dj + W]

    x = np.abs(gx)
    y = np.abs(gy) << 15
    t22 = x * cv3.TG22
    t67 = t22 + (x << 16)
    horiz = y < t22
    vert = ~horiz & (y > t67)
    diag = ~horiz & ~vert
    nmax = (horiz & (m > c(0, -1)) & (m >= c(0, 1))) | (vert & (m > c(-1, 0)) & (m >= c(1, 0)))
    dpos = (m > c(-1, -1)) & (m > c(1, 1))
    dneg = (m > c(-1, 1)) & (m > c(1, -1))
    nmax |= diag & np.where((gx ^ gy) < 0, dneg, dpos)
    cand = (m > lo) & nmax
    lab, _ = ndimage.label(cand, structure=np.ones((3, 3)))
    keep = np.zeros(lab.max() + 1, bool)
    keep[np.unique(lab[cand & (m > hi)])] = True
    keep[0] = False
    return np.where(keep[lab], 255, 0).astype(np.uint8)


def cv_canny(img, lo, hi, l2=False, aperture=3):
    """img: (H, W) or (H, W, C) uint8; returns the (H, W) uint8 0 / 255 map cv2.Canny(img, lo, hi, apertureSize=aperture,
    L2gradient=l2) gives.  Aperture 3 is oracle/cv_canny.py's restatement."""
    _check(aperture)
    if aperture == 3:
        return cv3.cv_canny(img, lo, hi, l2)
    dx, dy = cv_gradients(img, aperture)
    return canny_from_gradients(dx, dy, *cv_thresholds(lo, hi, l2, aperture), l2)
