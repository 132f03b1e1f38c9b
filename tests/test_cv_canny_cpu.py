"""CPU tests of the OpenCV-compatible path: the numpy restatement (oracle/cv_canny.py) against cv2.Canny, the argument and threshold
checks of b200_cv_canny_device_strided (they run before any device work) and the torch front end's rejections on CPU tensors."""
import ctypes as C
import math

import numpy as np
import pytest

import canny_edge_b200 as cb
from canny_edge_b200 import _lib
from oracle.cv_canny import cv_canny, cv_thresholds

IN, OUT = 1 << 32, 1 << 40   # device addresses far apart; never dereferenced by the checks


def _cv2():
    return pytest.importorskip("cv2")


def _image(rng, h, w, ch, kind):
    shape = (h, w) if ch == 1 else (h, w, ch)
    if kind == "noise":
        return rng.integers(0, 256, shape, dtype=np.uint8)
    if kind == "blocks":   # large flat regions with steps: long edges and ties
        by, bx = max(1, h // 6), max(1, w // 6)
        small = rng.integers(0, 256, (h // by + 1, w // bx + 1) + shape[2:], dtype=np.uint8)
        return np.ascontiguousarray(np.repeat(np.repeat(small, by, 0), bx, 1)[:h, :w])
    y, x = np.mgrid[0:h, 0:w]   # smooth ramps plus a little noise
    base = (x * rng.integers(1, 9) + y * rng.integers(1, 9)) % 256
    img = base[..., None] + rng.integers(-6, 7, (h, w, ch))
    img = np.clip(img, 0, 255).astype(np.uint8)
    return img[..., 0] if ch == 1 else img


def _thresholds(rng):
    kind = rng.integers(0, 6)
    if kind == 0:
        return float(rng.integers(0, 200)), float(rng.integers(50, 600))
    if kind == 1:   # swapped
        return float(rng.integers(300, 900)), float(rng.integers(0, 200))
    if kind == 2:   # fractional
        return float(rng.uniform(0, 300)), float(rng.uniform(100, 900))
    if kind == 3:   # negative
        return float(rng.uniform(-500, 10)), float(rng.uniform(-50, 400))
    if kind == 4:   # beyond any magnitude (L1 <= 2040; L2 thresholds are clamped to 32767)
        return float(rng.uniform(0, 100)), float(rng.choice([2041.0, 5000.0, 40000.0, 1e6]))
    return float(rng.integers(0, 100)), float(rng.integers(0, 100))


def test_restatement_equals_cv2_seeded():
    """320 seeded cases: 1 and 3 channels, L1 and L2, sizes from 1 x 1 to 90 x 90, every threshold family."""
    cv2 = _cv2()
    rng = np.random.default_rng(20261021)
    sizes = [(1, 1), (1, 7), (9, 1), (2, 2), (3, 5)]
    for i in range(320):
        h, w = sizes[i] if i < len(sizes) else (int(rng.integers(1, 91)), int(rng.integers(1, 91)))
        ch = 1 if i % 2 == 0 else 3
        l2 = (i // 2) % 2 == 1
        img = _image(rng, h, w, ch, ("noise", "blocks", "ramps")[i % 3])
        lo, hi = _thresholds(rng)
        want = cv2.Canny(img, lo, hi, L2gradient=l2)
        got = cv_canny(img, lo, hi, l2)
        assert np.array_equal(got, want), (i, h, w, ch, l2, lo, hi, int((got != want).sum()))


@pytest.mark.parametrize("h,w", [(1080, 1920), (2160, 3840)])
@pytest.mark.parametrize("ch", [1, 3])
def test_restatement_equals_cv2_large(h, w, ch):
    cv2 = _cv2()
    rng = np.random.default_rng(h + ch)
    img = _image(rng, h, w, ch, "blocks")
    img = np.clip(img.astype(np.int16) + rng.integers(-20, 21, img.shape), 0, 255).astype(np.uint8)
    for l2, (lo, hi) in ((False, (60.0, 180.0)), (True, (40.5, 120.25))):
        assert np.array_equal(cv_canny(img, lo, hi, l2), cv2.Canny(img, lo, hi, L2gradient=l2)), (l2, lo, hi)


def test_restatement_equals_cv2_on_a_strided_crop():
    cv2 = _cv2()
    rng = np.random.default_rng(7)
    big = _image(rng, 300, 400, 3, "noise")
    crop = big[17:250, 33:371]
    for l2 in (False, True):
        assert np.array_equal(cv_canny(crop, 100, 300, l2), cv2.Canny(crop, 100, 300, L2gradient=l2))
        assert np.array_equal(cv_canny(crop[..., 1], 50, 150, l2), cv2.Canny(np.ascontiguousarray(crop[..., 1]), 50, 150, L2gradient=l2))


def test_threshold_derivation():
    assert cv_thresholds(50.7, 20.2) == (20, 50)
    assert cv_thresholds(-3.5, 10.0) == (-4, 10)
    assert cv_thresholds(10.5, 20.0, l2=True) == (110, 400)
    assert cv_thresholds(-5.0, 1e9, l2=True) == (-5, 32767 * 32767)


def call(d_in=IN, in_pitch=None, in_fs=None, n=2, h=8, w=16, ch=1, t1=20.0, t2=60.0, l2=0, d_out=OUT, out_pitch=None, out_fs=None):
    lib = _lib.load()
    in_pitch = ch * w if in_pitch is None else in_pitch
    in_fs = h * in_pitch if in_fs is None else in_fs
    out_pitch = w if out_pitch is None else out_pitch
    out_fs = h * out_pitch if out_fs is None else out_fs
    return lib.b200_cv_canny_device_strided(None, d_in, in_pitch, in_fs, n, h, w, ch, C.c_double(t1), C.c_double(t2), l2, d_out,
                                            out_pitch, out_fs)


@pytest.mark.parametrize("ch", [1, 3])
def test_entry_point_rejects_bad_layouts(ch):
    h, w = 8, 16
    bad = {
        "null input": dict(d_in=None),
        "null output": dict(d_out=None),
        "height 0": dict(h=0),
        "width 0": dict(w=0),
        "no frames": dict(n=0),
        "negative input pitch": dict(in_pitch=-ch * w),
        "negative input frame stride": dict(in_fs=-1),
        "negative output pitch": dict(out_pitch=-w),
        "negative output frame stride": dict(out_fs=-1),
        "input pitch below a row": dict(in_pitch=ch * w - 1),
        "output pitch below a row": dict(out_pitch=w - 1),
        "input frames overlap": dict(in_fs=(h - 1) * ch * w + ch * w - 1),
        "output frames overlap": dict(out_fs=(h - 1) * w + w - 1),
        "broadcast input frames": dict(in_fs=0),
        "output inside the input": dict(d_out=IN + ch * w),
        "input inside the output": dict(d_in=OUT + w),
        "huge pitch": dict(in_pitch=(1 << 62) + 5),
        "huge frame stride": dict(n=1 << 30, in_fs=1 << 40),
    }
    for name, kw in bad.items():
        assert call(ch=ch, **kw) == _lib.ERR_INVALID_ARG, name
        assert _lib.load().b200_last_error(), name


def test_entry_point_checks_channels_and_thresholds():
    for ch in (0, 2, 4, -1):
        assert call(ch=ch, in_pitch=max(ch, 1) * 16) == _lib.ERR_UNSUPPORTED, ch
    for t1, t2 in ((math.nan, 10.0), (10.0, math.nan), (math.inf, 10.0), (10.0, -math.inf)):
        for l2 in (0, 1):
            assert call(t1=t1, t2=t2, l2=l2) == _lib.ERR_INVALID_ARG, (t1, t2, l2)
    # floors outside int32: OpenCV's cvFloor overflows there
    for t1, t2 in ((10.0, 1e10), (10.0, 2.0 ** 31), (-1e10, 10.0), (-(2.0 ** 31) - 1, 10.0)):
        assert call(t1=t1, t2=t2) == _lib.ERR_UNSUPPORTED, (t1, t2)
    assert call(t1=-1e10, t2=10.0, l2=1) == _lib.ERR_UNSUPPORTED   # negative L2 thresholds are not clamped
    assert call(n=1, h=65535 * 64 + 1, w=1) == _lib.ERR_UNSUPPORTED   # more rows than the kernel's grid covers
    # the channel check comes before the layout checks, the threshold checks before them too
    assert call(ch=2, d_in=None) == _lib.ERR_UNSUPPORTED
    assert call(t1=math.nan, d_in=None) == _lib.ERR_INVALID_ARG


def test_entry_point_accepts_good_arguments():
    """Valid calls pass every check and stop only at the missing device (B200_ERR_NO_DEVICE here, work on a GPU box)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: these fake addresses would be used")
    good = [
        {}, dict(ch=3), dict(h=1, w=1, n=1), dict(h=1, w=300), dict(h=300, w=1), dict(in_pitch=21, out_pitch=19),
        dict(n=1, in_fs=0, out_fs=0), dict(t1=300.0, t2=10.0), dict(t1=-5.5, t2=0.25), dict(t1=10.0, t2=1e10, l2=1),
        dict(t1=2.0 ** 31 - 1, t2=0.0), dict(l2=1, t1=1e300, t2=1e300),
    ]
    for kw in good:
        assert call(**kw) == _lib.ERR_NO_DEVICE, kw


def test_torch_front_end_rejections_on_cpu_tensors():
    import torch
    api = cb.torch_api
    x = torch.zeros((2, 32, 48), dtype=torch.uint8)
    with pytest.raises(ValueError, match="CUDA"):
        api.cv_canny(x, 20, 60)
    with pytest.raises(ValueError, match="CUDA"):
        api.cv_canny_color(torch.zeros((32, 48, 3), dtype=torch.uint8), 20, 60, L2gradient=True)
    with pytest.raises(ValueError, match="CUDA"):
        api.cv_canny(torch.zeros((1, 1), dtype=torch.uint8), 20, 60)   # 1 x 1 is a valid size; the device is not
    with pytest.raises(ValueError, match=r"\.contiguous\(\)"):
        api.cv_canny(x.transpose(1, 2), 20, 60)
    with pytest.raises(ValueError, match=r"\.contiguous\(\)"):
        api.cv_canny_color(torch.zeros((2, 3, 32, 48), dtype=torch.uint8).permute(0, 2, 3, 1), 20, 60)
    for t in (x.float(), x[..., None], torch.zeros((0, 5), dtype=torch.uint8), torch.zeros((4, 32, 48, 4), dtype=torch.uint8)):
        with pytest.raises(ValueError):
            api.cv_canny(t, 20, 60)
    for t in (x, torch.zeros((32, 48, 4), dtype=torch.uint8)):
        with pytest.raises(ValueError):
            api.cv_canny_color(t, 20, 60)
    # the 1-pixel minimum is the OpenCV calls' own: the reference-semantics calls keep theirs
    assert cb.torch_api.frame_layout(torch.zeros((1, 5), dtype=torch.uint8), min_side=1) == (1, 1, 5, 5, 5)
    with pytest.raises(ValueError, match="2 x 2"):
        cb.torch_api.frame_layout(torch.zeros((1, 5), dtype=torch.uint8))
