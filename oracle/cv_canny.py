"""TEST INFRASTRUCTURE ONLY: cv::Canny (OpenCV 4.x, apertureSize = 3) restated in numpy, bit for bit.

The specification of b200_cv_canny_device_strided.  Plain numpy plus scipy.ndimage.label, so the GPU tests do not need cv2.
Checked against cv2.Canny by tests/test_cv_canny_cpu.py wherever cv2 is importable.

    Sobel 3x3 with BORDER_REPLICATE on every channel; per pixel the channel of largest magnitude (the first on ties), magnitude
    |dx|+|dy| (L1) or dx^2+dy^2 (L2, against squared thresholds); direction by the fixed-point tan(22.5 deg) test; non-maximum
    suppression with `>` on one side and `>=` on the other (both `>` on diagonals); `> low` candidates, `> high` seeds; plain
    8-connected hysteresis.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage

TG22 = int(0.4142135623730950488016887242097 * (1 << 15) + 0.5)   # 13573


def cv_thresholds(lo: float, hi: float, l2: bool = False):
    """(low, high) as integers in magnitude space, as cv::Canny derives them (swapped when low > high, clamped and squared for
    L2, floored)."""
    if lo > hi:
        lo, hi = hi, lo
    if l2:
        lo, hi = min(32767.0, lo), min(32767.0, hi)
        if lo > 0:
            lo *= lo
        if hi > 0:
            hi *= hi
    return int(np.floor(lo)), int(np.floor(hi))


def cv_canny(img, lo, hi, l2=False):
    """img: (H, W) or (H, W, C) uint8; returns the (H, W) uint8 0 / 255 map cv2.Canny(img, lo, hi, L2gradient=l2) gives."""
    img = np.asarray(img).astype(np.int32)
    if img.ndim == 2:
        img = img[..., None]
    H, W, C = img.shape
    p = np.pad(img, ((1, 1), (1, 1), (0, 0)), mode="edge")                  # BORDER_REPLICATE
    dx = (p[:-2, 2:] - p[:-2, :-2]) + 2 * (p[1:-1, 2:] - p[1:-1, :-2]) + (p[2:, 2:] - p[2:, :-2])
    dy = (p[2:, :-2] - p[:-2, :-2]) + 2 * (p[2:, 1:-1] - p[:-2, 1:-1]) + (p[2:, 2:] - p[:-2, 2:])
    n = dx * dx + dy * dy if l2 else np.abs(dx) + np.abs(dy)
    k = np.argmax(n, axis=2)                                                 # first channel of maximal magnitude
    ii, jj = np.indices((H, W))
    m, gx, gy = n[ii, jj, k], dx[ii, jj, k], dy[ii, jj, k]
    lo, hi = cv_thresholds(lo, hi, l2)
    M = np.pad(m, 1)                                                         # magnitude outside the image is 0

    def c(di, dj):
        return M[1 + di:1 + di + H, 1 + dj:1 + dj + W]

    x = np.abs(gx).astype(np.int64)
    y = np.abs(gy).astype(np.int64) << 15
    t22 = x * TG22
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
