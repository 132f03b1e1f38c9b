"""CPU tests of cv::Canny's apertureSize 5 and 7: the numpy restatement (tests/cv_canny_aperture_ref.py) against cv2.Canny, the
argument checks of b200_cv_canny_aperture_device_strided and b200_cv_canny_aperture_frames_device (they run before any device work,
in a fixed order) and the torch front end's apertureSize on CPU tensors."""
import ctypes as C
import math

import numpy as np
import pytest

import canny_edge_b200 as cb
from canny_edge_b200 import _lib
from canny_edge_b200.api import frame_list
from cv_canny_aperture_ref import canny_from_gradients, cv_canny, cv_gradients, cv_thresholds, sobel_sums
from oracle import cv_canny as cv3
from test_cv_canny_cpu import _image, _thresholds
from test_cv_ragged_cpu import desc

IN, OUT = 1 << 32, 1 << 40   # device addresses far apart; never dereferenced by the checks
BAD_APERTURES = (1, 2, 4, 6, 8, 9, 0, -1)
# magnitudes grow about 16x over aperture 3 at apertures 5 and 7 (7 after its 1/16, which also divides its thresholds): half of
# the seeded cases scale their thresholds so that every family still lands among the magnitudes
SCALE = {3: 1.0, 5: 16.0, 7: 16.0 * 16.0}


def _cv2():
    return pytest.importorskip("cv2")


def _corpus(aperture, n=320, seed=20261021):
    """n seeded cases: 1 and 3 channels, L1 and L2, sizes from 1 x 1 to 90 x 90 (1 x N, N x 1 and frames narrower than the kernel
    first), noise / blocks / ramps, every threshold family of test_cv_canny_cpu.py, half of them scaled to the aperture."""
    rng = np.random.default_rng(seed + aperture)
    sizes = [(1, 1), (1, 7), (9, 1), (2, 2), (3, 5), (5, 3), (6, 6), (1, 90), (90, 1)]
    for i in range(n):
        h, w = sizes[i] if i < len(sizes) else (int(rng.integers(1, 91)), int(rng.integers(1, 91)))
        ch = 1 if i % 2 == 0 else 3
        l2 = (i // 2) % 2 == 1
        img = _image(rng, h, w, ch, ("noise", "blocks", "ramps")[i % 3])
        lo, hi = _thresholds(rng)
        if (i // 4) % 2:
            lo, hi = lo * SCALE[aperture], hi * SCALE[aperture]
        yield i, img, lo, hi, l2


@pytest.mark.parametrize("aperture", [3, 5, 7])
def test_restatement_equals_cv2_seeded(aperture):
    cv2 = _cv2()
    for i, img, lo, hi, l2 in _corpus(aperture):
        want = cv2.Canny(img, lo, hi, apertureSize=aperture, L2gradient=l2)
        got = cv_canny(img, lo, hi, l2, aperture)
        assert np.array_equal(got, want), (i, img.shape, l2, lo, hi, int((got != want).sum()))


def test_aperture_3_gradients_are_oracle_cv_canny():
    """The generic separable gradients at aperture 3 give oracle/cv_canny.py's maps: the wider apertures share its rules."""
    for i, img, lo, hi, l2 in _corpus(3, n=60):
        dx, dy = cv_gradients(img, 3)
        assert np.array_equal(canny_from_gradients(dx, dy, *cv_thresholds(lo, hi, l2, 3), l2), cv3.cv_canny(img, lo, hi, l2)), i


def test_half_to_even_rounding_matters():
    """Aperture 7 rounds S / 16 half to even (cvRound).  Half-up rounding is wrong, and the corpus shows it: some of its cases
    change under half-up rounding, and those still match cv2 with half to even."""
    changed = 0
    for i, img, lo, hi, l2 in _corpus(7):
        sx, sy = sobel_sums(img, 7)
        if not ((sx % 16 == 8).any() or (sy % 16 == 8).any()):
            continue
        up = canny_from_gradients((sx + 8) >> 4, (sy + 8) >> 4, *cv_thresholds(lo, hi, l2, 7), l2)
        changed += not np.array_equal(up, cv_canny(img, lo, hi, l2, 7))
    assert changed >= 1
    # a 40 x 50 noise image: many exact halves
    img = np.random.default_rng(4050).integers(0, 256, (40, 50), dtype=np.uint8)
    sx, sy = sobel_sums(img, 7)
    assert (sx % 16 == 8).sum() + (sy % 16 == 8).sum() > 50
    assert np.array_equal(_rint16(sx), cv_gradients(img, 7)[0])


def _rint16(s):
    """np.rint (round half to even) of s / 16, which is exact in float64 for these sums."""
    return np.rint(s / 16.0).astype(np.int64)


@pytest.mark.parametrize("aperture", [5, 7])
@pytest.mark.parametrize("h,w", [(1080, 1920), (2160, 3840)])
@pytest.mark.parametrize("ch", [1, 3])
def test_restatement_equals_cv2_large(aperture, h, w, ch):
    cv2 = _cv2()
    rng = np.random.default_rng(h + ch + aperture)
    img = _image(rng, h, w, ch, "blocks")
    img = np.clip(img.astype(np.int16) + rng.integers(-20, 21, img.shape), 0, 255).astype(np.uint8)
    s = SCALE[aperture]
    for l2, (lo, hi) in ((False, (60.0 * s, 180.0 * s)), (True, (40.5 * s, 120.25 * s))):
        want = cv2.Canny(img, lo, hi, apertureSize=aperture, L2gradient=l2)
        assert want.any() and not want.all()
        assert np.array_equal(cv_canny(img, lo, hi, l2, aperture), want), (l2, lo, hi)


@pytest.mark.parametrize("aperture", [5, 7])
def test_restatement_equals_cv2_on_a_strided_crop(aperture):
    cv2 = _cv2()
    rng = np.random.default_rng(7)
    big = _image(rng, 300, 400, 3, "noise")
    crop = big[17:250, 33:371]
    s = SCALE[aperture]
    for l2 in (False, True):
        assert np.array_equal(cv_canny(crop, 100 * s, 300 * s, l2, aperture),
                              cv2.Canny(crop, 100 * s, 300 * s, apertureSize=aperture, L2gradient=l2))
        gray = crop[..., 1]
        assert np.array_equal(cv_canny(gray, 50 * s, 150 * s, l2, aperture),
                              cv2.Canny(np.ascontiguousarray(gray), 50 * s, 150 * s, apertureSize=aperture, L2gradient=l2))


def test_aperture_7_thresholds_against_cv2():
    """Aperture 7 divides the thresholds by 16 before the L2 clamp and the floor."""
    cv2 = _cv2()
    img = np.random.default_rng(64).integers(0, 256, (64, 64), dtype=np.uint8)
    # 600000 / 16 = 37500 is clamped to 32767, whose square is above any magnitude: no edges (clamping first would give some)
    want = cv2.Canny(img, 10, 600000, apertureSize=7, L2gradient=True)
    assert not want.any()
    assert np.array_equal(cv_canny(img, 10, 600000, True, 7), want)
    assert canny_from_gradients(*cv_gradients(img, 7), *cv3.cv_thresholds(10 / 16, 32767 / 16, True), True).any()
    # 2^34 / 16 = 2^30 fits in int32: accepted, above every magnitude
    want = cv2.Canny(img, 2.0 ** 34, 2.0 ** 34, apertureSize=7)
    assert not want.any()
    assert np.array_equal(cv_canny(img, 2.0 ** 34, 2.0 ** 34, False, 7), want)


def test_threshold_derivation_aperture_7():
    assert cv_thresholds(160.0, 480.0, aperture=7) == (10, 30)
    assert cv_thresholds(170.0, 100.0, aperture=7) == (6, 10)          # divided, then swapped, then floored
    assert cv_thresholds(-81.0, 8.0, aperture=7) == (-6, 0)
    assert cv_thresholds(10.0, 600000.0, l2=True, aperture=7) == (0, 32767 * 32767)   # 0.625^2 floors to 0
    assert cv_thresholds(40.0, 160.0, l2=True, aperture=7) == (6, 100)
    assert cv_thresholds(0.0, 2.0 ** 34, aperture=7) == (0, 1 << 30)
    assert cv_thresholds(160.0, 480.0, aperture=5) == (160, 480)
    assert cv_thresholds(160.0, 480.0, l2=True, aperture=5) == cv3.cv_thresholds(160.0, 480.0, True)
    with pytest.raises(ValueError):
        cv_thresholds(1.0, 2.0, aperture=4)


# ---- the C calls ----------------------------------------------------------------------------------------------------------------

def call(d_in=IN, in_pitch=None, in_fs=None, n=2, h=8, w=16, ch=1, t1=20.0, t2=60.0, aperture=5, l2=0, d_out=OUT, out_pitch=None,
         out_fs=None):
    in_pitch = ch * w if in_pitch is None else in_pitch
    in_fs = h * in_pitch if in_fs is None else in_fs
    out_pitch = w if out_pitch is None else out_pitch
    out_fs = h * out_pitch if out_fs is None else out_fs
    return _lib.load().b200_cv_canny_aperture_device_strided(None, d_in, in_pitch, in_fs, n, h, w, ch, C.c_double(t1), C.c_double(t2),
                                                             aperture, l2, d_out, out_pitch, out_fs)


def call_list(descs, ch=1, t1=20.0, t2=60.0, aperture=5, l2=0, n=None):
    return _lib.load().b200_cv_canny_aperture_frames_device(None, frame_list(descs), len(descs) if n is None else n, ch, C.c_double(t1),
                                                            C.c_double(t2), aperture, l2)


def no_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: these fake addresses would be used")


@pytest.mark.parametrize("ch", [1, 3])
def test_bad_apertures_are_invalid(ch):
    for a in BAD_APERTURES:
        for l2 in (0, 1):
            assert call(ch=ch, aperture=a, l2=l2) == _lib.ERR_INVALID_ARG, a
            assert b"aperture" in _lib.load().b200_last_error()
            assert call_list([desc(0, ch=ch)], ch, aperture=a, l2=l2) == _lib.ERR_INVALID_ARG, a
            assert b"aperture" in _lib.load().b200_last_error()


def test_check_order():
    """channels, then aperture, then (uniform call) height, then thresholds, then the layout / list."""
    for bad_ch in (0, 2, 4):
        assert call(ch=bad_ch, aperture=4) == _lib.ERR_UNSUPPORTED
        assert call_list([desc(0)], bad_ch, aperture=4) == _lib.ERR_UNSUPPORTED
    for a in (4, 9):
        assert call(aperture=a, n=1, h=65535 * 64 + 1, w=1) == _lib.ERR_INVALID_ARG
        assert call(aperture=a, t1=math.nan) == _lib.ERR_INVALID_ARG
        assert b"aperture" in _lib.load().b200_last_error()
        assert call(aperture=a, t1=1e12) == _lib.ERR_INVALID_ARG
        assert call_list([desc(0)], aperture=a, t1=1e12) == _lib.ERR_INVALID_ARG
        assert b"aperture" in _lib.load().b200_last_error()
    for a in (3, 5, 7):
        assert call(aperture=a, n=1, h=65535 * 64 + 1, w=1, t1=math.nan) == _lib.ERR_UNSUPPORTED
        assert call(aperture=a, t1=math.nan, d_in=None) == _lib.ERR_INVALID_ARG
        assert b"finite" in _lib.load().b200_last_error()
        assert call(aperture=a, t1=2.0 ** 40, d_in=None) == _lib.ERR_UNSUPPORTED
        assert call_list([desc(0, d_in=0)], aperture=a, t1=2.0 ** 40) == _lib.ERR_UNSUPPORTED
        assert call_list([desc(0, d_in=0)], aperture=a, t1=math.inf) == _lib.ERR_INVALID_ARG
        assert b"finite" in _lib.load().b200_last_error()
        assert call(aperture=a, d_in=None) == _lib.ERR_INVALID_ARG
        assert call_list([desc(0, d_in=0)], aperture=a) == _lib.ERR_INVALID_ARG


def test_aperture_7_threshold_range():
    """The int32 check applies to the threshold divided by 16: 2^34 is accepted, 2^35 (2^31 after the division) is not."""
    for t in (2.0 ** 35, -(2.0 ** 35) - 16):
        assert call(aperture=7, t2=t) == _lib.ERR_UNSUPPORTED, t
        assert call_list([desc(0)], aperture=7, t2=t) == _lib.ERR_UNSUPPORTED, t
    for a in (3, 5):
        assert call(aperture=a, t2=2.0 ** 34) == _lib.ERR_UNSUPPORTED
        assert call_list([desc(0)], aperture=a, t2=2.0 ** 34) == _lib.ERR_UNSUPPORTED
    no_gpu()
    for t in (2.0 ** 34, -(2.0 ** 35), 2.0 ** 35 - 17):
        assert call(aperture=7, t2=t) == _lib.ERR_NO_DEVICE, t
        assert call_list([desc(0)], aperture=7, t2=t) == _lib.ERR_NO_DEVICE, t


@pytest.mark.parametrize("aperture", [3, 5, 7])
def test_good_arguments_reach_the_device(aperture):
    """The good-argument cases of the aperture-3 CPU tests pass every check and stop only at the missing device."""
    no_gpu()
    good = [
        {}, dict(ch=3), dict(h=1, w=1, n=1), dict(h=1, w=300), dict(h=300, w=1), dict(in_pitch=21, out_pitch=19),
        dict(n=1, in_fs=0, out_fs=0), dict(t1=300.0, t2=10.0), dict(t1=-5.5, t2=0.25), dict(t1=10.0, t2=1e10, l2=1),
        dict(t1=2.0 ** 31 - 1, t2=0.0), dict(l2=1, t1=1e300, t2=1e300), dict(h=2, w=2, n=1), dict(h=3, w=5, n=1),
    ]
    for kw in good:
        assert call(aperture=aperture, **kw) == _lib.ERR_NO_DEVICE, kw
    for ch in (1, 3):
        lists = [
            [desc(0, ch=ch)], [desc(0, h=1, w=1, ch=ch)], [desc(0, h=2, w=2, ch=ch), desc(1, h=3, w=5, ch=ch)],
            [desc(0, h=1, w=37, ch=ch), desc(1, h=45, w=1, ch=ch)], [desc(0, ch=ch, in_pitch=ch * 16 + 5, out_pitch=19)],
            [desc(0, h=5_000_000, w=1, ch=ch, in_pitch=ch)], [desc(i, h=1 + i, w=1 + 3 * i, ch=ch) for i in range(20)],
        ]
        for descs in lists:
            assert call_list(descs, ch, aperture=aperture) == _lib.ERR_NO_DEVICE, descs[:2]
        for t1, t2, l2 in ((60, 20, 0), (-5, -1, 0), (0, 0, 1), (1e9, 1e9, 1), (2.0 ** 31 - 1, 0, 0)):
            assert call_list([desc(0, ch=ch)], ch, t1, t2, aperture, l2) == _lib.ERR_NO_DEVICE, (t1, t2, l2)


def test_ctypes_entries_and_python_wrappers():
    for name in ("b200_cv_canny_aperture_device_strided", "b200_cv_canny_aperture_frames_device"):
        assert name in _lib.SIGNATURES
    assert _lib.load().b200_version() == 1
    import inspect
    for fn in (cb.cv_canny_device_strided_ptr, cb.cv_canny_frames_device_ptr):
        assert inspect.signature(fn).parameters["aperture_size"].default == 3
    for fn in (cb.torch_api.cv_canny, cb.torch_api.cv_canny_color, cb.torch_api.cv_canny_list, cb.torch_api.cv_canny_color_list):
        p = inspect.signature(fn).parameters["apertureSize"]
        assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default == 3


def test_python_wrappers_raise_c_errors():
    """A bad aperture reaches the C check through the Python wrappers and raises like any other C argument error."""
    with pytest.raises(_lib.CannyB200Error, match="aperture"):
        cb.cv_canny_device_strided_ptr(None, IN, 16, 128, 2, 8, 16, 1, 20, 60, False, OUT, 16, 128, aperture_size=4)
    with pytest.raises(_lib.CannyB200Error, match="aperture"):
        cb.cv_canny_frames_device_ptr(None, [desc(0)], 1, 20, 60, True, aperture_size=9)


def test_torch_front_end_rejections_on_cpu_tensors():
    import torch
    api = cb.torch_api
    x = torch.zeros((2, 32, 48), dtype=torch.uint8)
    c = torch.zeros((32, 48, 3), dtype=torch.uint8)
    for a in (3, 5, 7, 4, 0):
        with pytest.raises(ValueError, match="CUDA"):
            api.cv_canny(x, 20, 60, apertureSize=a)
        with pytest.raises(ValueError, match="CUDA"):
            api.cv_canny_color(c, 20, 60, apertureSize=a, L2gradient=True)
        with pytest.raises(ValueError, match="CUDA"):
            api.cv_canny_list([x[0], x[1, :5, :7]], 20, 60, apertureSize=a)
        with pytest.raises(ValueError, match="CUDA"):
            api.cv_canny_color_list([c], 20, 60, apertureSize=a)
    with pytest.raises(TypeError):
        api.cv_canny(x, 20, 60, 5)   # keyword-only, as the other cv2 options
    with pytest.raises((TypeError, ValueError)):
        api.cv_canny(x, 20, 60, apertureSize="five")
