"""CPU tests of the Gaussian pre-blur of the OpenCV-compatible path: the numpy restatement (tests/cv_gaussian_ref.py) against
cv2.GaussianBlur and cv2.Canny(cv2.GaussianBlur(...)), b200_cv_gaussian_kernel against the restatement, the argument checks of
b200_cv_gaussian_canny_device_strided and b200_cv_gaussian_canny_frames_device (they run before any device work, in a fixed order)
and the torch front end's gaussian= on CPU tensors."""
import ctypes as C
import math

import numpy as np
import pytest

import canny_edge_b200 as cb
from canny_edge_b200 import _lib
from canny_edge_b200.api import frame_list
from cv_canny_aperture_ref import cv_canny
from cv_gaussian_ref import GaussArgError, cv2_gaussian_blur, fixed_taps, gaussian_blur, kernel, resolve
from test_cv_canny_cpu import _image, _thresholds
from test_cv_ragged_cpu import desc

IN, OUT = 1 << 32, 1 << 40   # device addresses far apart; never dereferenced by the checks
SCALE = {3: 1.0, 5: 16.0, 7: 16.0 * 16.0}


def _cv2():
    return pytest.importorskip("cv2")


def _blur_args(rng, i):
    """One argument family per case: the sigma-0 tables, explicit sigma, derived ksize, asymmetric ksize and sigmas, negative sigma,
    (1, 1), and sides up to 31."""
    fam = i % 7
    if fam == 0:
        k = int(rng.choice([1, 3, 5, 7]))
        return (k, k), 0.0, 0.0
    if fam == 1:
        k = int(rng.choice([3, 5, 7, 9, 11, 15, 21, 31]))
        return (k, k), float(rng.uniform(0.05, 6.0)), 0.0
    if fam == 2:
        return (0, 0), float(np.round(rng.uniform(0.1, 5.0), 2)), 0.0
    if fam == 3:
        kw, kh = int(rng.choice([1, 3, 5, 9, 13, 31])), int(rng.choice([1, 3, 7, 11, 25]))
        return (kw, kh), float(rng.uniform(0.0, 5.0)), float(rng.choice([0.0, rng.uniform(0.1, 5.0)]))
    if fam == 4:
        k = int(rng.choice([3, 5, 7, 9]))
        return (k, k), float(rng.uniform(-3.0, -0.01)), float(rng.choice([0.0, -1.0]))
    if fam == 5:
        return (1, 1), float(rng.uniform(0, 3)), 0.0
    return (int(rng.choice([9, 11, 13, 21, 31])), int(rng.choice([3, 9, 15, 31]))), 0.0, 0.0


def _corpus(n=420, seed=20261022):
    """n seeded cases: 1 and 3 channels, sizes from 1 x 1 to 70 x 70 (1 x N, N x 1 and frames smaller than the kernel first),
    noise / blocks / ramps, every blur family, apertures 3 / 5 / 7 with thresholds scaled to them, L1 and L2."""
    rng = np.random.default_rng(seed)
    sizes = [(1, 1), (1, 9), (11, 1), (2, 2), (3, 5), (5, 3), (1, 40), (40, 1), (4, 31), (31, 4)]
    for i in range(n):
        h, w = sizes[i] if i < len(sizes) else (int(rng.integers(1, 71)), int(rng.integers(1, 71)))
        ch = 1 if i % 2 == 0 else 3
        img = _image(rng, h, w, ch, ("noise", "blocks", "ramps")[i % 3])
        ksize, sx, sy = _blur_args(rng, i)
        aperture = (3, 5, 7)[(i // 2) % 3]
        l2 = (i // 6) % 2 == 1
        lo, hi = _thresholds(rng)
        if (i // 12) % 2:
            lo, hi = lo * SCALE[aperture], hi * SCALE[aperture]
        yield i, img, ksize, sx, sy, aperture, l2, lo, hi


def test_blur_restatement_equals_cv2_seeded():
    cv2 = _cv2()
    for i, img, ksize, sx, sy, *_ in _corpus():
        want = cv2_gaussian_blur(cv2, img, ksize, sx, sy)
        got = gaussian_blur(img, ksize, sx, sy)
        assert np.array_equal(got, want), (i, img.shape, ksize, sx, sy, int((got != want).sum()))


def test_canny_of_blur_equals_cv2_seeded():
    cv2 = _cv2()
    for i, img, ksize, sx, sy, aperture, l2, lo, hi in _corpus():
        want = cv2.Canny(cv2_gaussian_blur(cv2, img, ksize, sx, sy), lo, hi, apertureSize=aperture, L2gradient=l2)
        got = cv_canny(gaussian_blur(img, ksize, sx, sy), lo, hi, l2, aperture)
        assert np.array_equal(got, want), (i, img.shape, ksize, sx, sy, aperture, l2, lo, hi)


@pytest.mark.parametrize("args", [((5, 5), 0.0, 0.0), ((0, 0), 1.4, 0.0), ((0, 0), 2.0, 0.0), ((31, 31), 0.0, 0.0),
                                  ((0, 0), 5.0, 0.0), ((31, 7), 3.0, 1.1)])
def test_blur_restatement_equals_cv2_4k(args):
    cv2 = _cv2()
    rng = np.random.default_rng(2160)
    img = _image(rng, 2160, 3840, 3, "blocks")
    img = np.clip(img.astype(np.int16) + rng.integers(-20, 21, img.shape), 0, 255).astype(np.uint8)
    crop = img[13:2001, 7:3331]
    for src in (img, crop, np.ascontiguousarray(img[..., 1])):
        assert np.array_equal(gaussian_blur(src, *args), cv2_gaussian_blur(cv2, src, *args)), args


def test_canny_of_blur_equals_cv2_1080p():
    cv2 = _cv2()
    rng = np.random.default_rng(1080)
    img = _image(rng, 1080, 1920, 1, "blocks")
    img = np.clip(img.astype(np.int16) + rng.integers(-40, 41, img.shape), 0, 255).astype(np.uint8)
    for ksize, s in (((5, 5), 0.0), ((0, 0), 1.4), ((31, 31), 0.0)):
        want = cv2.Canny(cv2_gaussian_blur(cv2, img, ksize, s), 20, 60)
        assert want.any()
        assert np.array_equal(cv_canny(gaussian_blur(img, ksize, s), 20, 60), want), ksize


def test_resolution_rules():
    assert resolve((0, 0), 1.4) == ((9, 9), 1.4, 1.4)
    assert resolve((0, 0), 2.0)[0] == (13, 13)
    assert resolve((0, 0), 5.0)[0] == (31, 31)
    assert resolve((0, 5), 0.5, 0.0)[0] == (5, 5)                     # sigmaY 0 takes sigmaX
    assert resolve((0, 0), 1.4, 2.0)[0] == (9, 13)
    assert resolve((5, 5), -1.0) == ((5, 5), 0.0, 0.0)                # negative sigma: 0 after the derivation
    assert resolve((0, 0), 0.25)[0] == (3, 3)                         # cvRound(2.5) = 2, | 1
    assert resolve((0, 0), 0.75)[0] == (7, 7)                         # cvRound(5.5) = 6, | 1
    assert resolve((5, -3), 1.0)[0] == (5, 7)                         # a negative side is derived too
    for ksize, s in (((0, 0), 0.0), ((4, 4), 1.0), ((0, 5), 0.0), ((5, -3), 0.0), ((0, 0), -2.0)):
        with pytest.raises(GaussArgError) as e:
            resolve(ksize, s)
        assert e.value.status == _lib.ERR_INVALID_ARG
    for ksize, s in (((33, 33), 0.0), ((0, 0), 5.1), ((3, 45), 1.0)):
        with pytest.raises(GaussArgError) as e:
            resolve(ksize, s)
        assert e.value.status == _lib.ERR_UNSUPPORTED


def test_fixed_point_tables():
    assert list(fixed_taps(7, 0.0)) == [8, 28, 56, 72, 56, 28, 8]
    assert list(fixed_taps(5, 0.0)) == [16, 64, 96, 64, 16]
    assert list(fixed_taps(3, 0.0)) == [64, 128, 64]
    assert list(fixed_taps(1, 0.0)) == [256]
    assert list(fixed_taps(3, 0.1)) == [0, 256, 0]
    for n in range(1, 32, 2):
        for s in (0.0, 0.3, 1.0, 4.0):
            f = fixed_taps(n, s)
            assert f.sum() == 256 and (f >= 0).all() and list(f) == list(f[::-1]), (n, s)


# ---- the C calls ----------------------------------------------------------------------------------------------------------------

def test_kernel_taps_equal_the_restatement():
    """b200_cv_gaussian_kernel (the taps the front kernel uses) equals the restatement for every odd size 1 .. 31 over a dense
    sigma grid, and for derived sizes; libm's exp in both is the evidence that OpenCV's softfloat exp is matched."""
    sigmas = [0.0] + [round(0.05 + 0.01 * i, 2) for i in range(496)]
    for n in range(1, 32, 2):
        for s in sigmas:
            got = cb.cv_gaussian_kernel(n, s)
            assert np.array_equal(got, fixed_taps(n, s)), (n, s, got)
    for s in sigmas[1:] + [-1.0]:
        try:
            want = kernel(0, s)
        except GaussArgError as e:
            with pytest.raises(_lib.CannyB200Error) as ce:
                cb.cv_gaussian_kernel(0, s)
            assert ce.value.status == e.status, s
            continue
        got = cb.cv_gaussian_kernel(0, s)
        assert len(got) == want[0] and np.array_equal(got, want[1]), s


def test_kernel_taps_against_cv2():
    """The double taps before the fixed-point step agree with cv2.getGaussianKernel's (whose sigma-0 path has a table of its own
    for n = 9, so sigma 0 is compared up to n = 7 only)."""
    cv2 = _cv2()
    from cv_gaussian_ref import kernel_bitexact
    for n in range(1, 32, 2):
        for s in (0.0, 0.6, 1.4, 2.0, 3.3, 5.0):
            if s == 0.0 and n > 7:
                continue
            want = cv2.getGaussianKernel(n, s, cv2.CV_64F).ravel()
            assert np.allclose(kernel_bitexact(n, s), want, rtol=0, atol=1e-15), (n, s)


def test_kernel_rejections():
    lib = _lib.load()
    n = C.c_int(0)
    taps = (C.c_int32 * 31)()
    for k, s, code in ((0, 0.0, _lib.ERR_INVALID_ARG), (4, 1.0, _lib.ERR_INVALID_ARG), (-3, 0.0, _lib.ERR_INVALID_ARG),
                       (5, math.nan, _lib.ERR_INVALID_ARG), (0, math.inf, _lib.ERR_INVALID_ARG), (33, 1.0, _lib.ERR_UNSUPPORTED),
                       (0, 5.1, _lib.ERR_UNSUPPORTED), (0, 1e300, _lib.ERR_UNSUPPORTED)):
        assert lib.b200_cv_gaussian_kernel(k, C.c_double(s), C.byref(n), taps) == code, (k, s)
    assert lib.b200_cv_gaussian_kernel(5, C.c_double(1.0), None, taps) == _lib.ERR_INVALID_ARG
    assert lib.b200_cv_gaussian_kernel(5, C.c_double(1.0), C.byref(n), None) == _lib.ERR_INVALID_ARG
    assert lib.b200_cv_gaussian_kernel(0, C.c_double(5.0), C.byref(n), taps) == _lib.OK and n.value == 31


def call(d_in=IN, in_pitch=None, in_fs=None, n=2, h=8, w=16, ch=1, ksize=(5, 5), sx=0.0, sy=0.0, t1=20.0, t2=60.0, aperture=3,
         l2=0, d_out=OUT, out_pitch=None, out_fs=None):
    in_pitch = ch * w if in_pitch is None else in_pitch
    in_fs = h * in_pitch if in_fs is None else in_fs
    out_pitch = w if out_pitch is None else out_pitch
    out_fs = h * out_pitch if out_fs is None else out_fs
    return _lib.load().b200_cv_gaussian_canny_device_strided(None, d_in, in_pitch, in_fs, n, h, w, ch, ksize[0], ksize[1],
                                                             C.c_double(sx), C.c_double(sy), C.c_double(t1), C.c_double(t2),
                                                             aperture, l2, d_out, out_pitch, out_fs)


def call_list(descs, ch=1, ksize=(5, 5), sx=0.0, sy=0.0, t1=20.0, t2=60.0, aperture=3, l2=0):
    return _lib.load().b200_cv_gaussian_canny_frames_device(None, frame_list(descs), len(descs), ch, ksize[0], ksize[1],
                                                            C.c_double(sx), C.c_double(sy), C.c_double(t1), C.c_double(t2),
                                                            aperture, l2)


def no_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: these fake addresses would be used")


BAD_BLURS = [((0, 0), 0.0, 0.0, _lib.ERR_INVALID_ARG), ((4, 4), 1.0, 0.0, _lib.ERR_INVALID_ARG),
             ((0, 5), 0.0, 0.0, _lib.ERR_INVALID_ARG), ((5, 0), 0.0, 0.0, _lib.ERR_INVALID_ARG),
             ((-1, 3), 0.0, 0.0, _lib.ERR_INVALID_ARG), ((5, 5), math.nan, 0.0, _lib.ERR_INVALID_ARG),
             ((5, 5), 1.0, math.inf, _lib.ERR_INVALID_ARG), ((5, 5), -math.inf, 0.0, _lib.ERR_INVALID_ARG),
             ((33, 3), 0.0, 0.0, _lib.ERR_UNSUPPORTED), ((3, 45), 0.0, 0.0, _lib.ERR_UNSUPPORTED),
             ((0, 0), 5.1, 0.0, _lib.ERR_UNSUPPORTED), ((0, 0), 1.0, 6.0, _lib.ERR_UNSUPPORTED),
             ((0, 0), 1e300, 0.0, _lib.ERR_UNSUPPORTED)]


@pytest.mark.parametrize("ch", [1, 3])
def test_bad_blur_arguments(ch):
    for ksize, sx, sy, code in BAD_BLURS:
        assert call(ch=ch, ksize=ksize, sx=sx, sy=sy) == code, (ksize, sx, sy)
        assert call_list([desc(0, ch=ch)], ch, ksize, sx, sy) == code, (ksize, sx, sy)


def test_check_order():
    """channels (UNSUPPORTED), aperture (INVALID_ARG), blur (INVALID_ARG before UNSUPPORTED), then (uniform call) height, thresholds,
    layout / list."""
    for bad_ch in (0, 2, 4):
        assert call(ch=bad_ch, aperture=4, ksize=(4, 4)) == _lib.ERR_UNSUPPORTED
        assert call_list([desc(0)], bad_ch, (4, 4), aperture=4) == _lib.ERR_UNSUPPORTED
    # aperture before the blur
    assert call(aperture=4, ksize=(33, 33)) == _lib.ERR_INVALID_ARG
    assert b"aperture" in _lib.load().b200_last_error()
    assert call_list([desc(0)], aperture=9, ksize=(33, 33)) == _lib.ERR_INVALID_ARG
    assert b"aperture" in _lib.load().b200_last_error()
    # within the blur: an invalid side before an unsupported one
    assert call(ksize=(33, 4)) == _lib.ERR_INVALID_ARG
    assert call(ksize=(33, 3), sx=math.nan) == _lib.ERR_INVALID_ARG
    assert call_list([desc(0)], ksize=(4, 45)) == _lib.ERR_INVALID_ARG
    # the blur before the height, the thresholds and the layout
    for ksize, sx, sy, code in BAD_BLURS:
        assert call(ksize=ksize, sx=sx, sy=sy, n=1, h=65535 * 64 + 1, w=1, t1=math.nan, d_in=None) == code
        assert b"Gaussian" in _lib.load().b200_last_error()
        assert call_list([desc(0, d_in=0)], ksize=ksize, sx=sx, sy=sy, t1=math.nan) == code
        assert b"Gaussian" in _lib.load().b200_last_error()
    # with a good blur, the existing checks in their order
    for ksize, sx in (((5, 5), 0.0), ((0, 0), 1.4), ((31, 31), 0.0), ((1, 1), 0.0)):
        assert call(ksize=ksize, sx=sx, n=1, h=65535 * 64 + 1, w=1, t1=math.nan) == _lib.ERR_UNSUPPORTED
        assert call(ksize=ksize, sx=sx, t1=math.nan, d_in=None) == _lib.ERR_INVALID_ARG
        assert b"finite" in _lib.load().b200_last_error()
        assert call(ksize=ksize, sx=sx, t1=2.0 ** 40, d_in=None) == _lib.ERR_UNSUPPORTED
        assert call(ksize=ksize, sx=sx, d_in=None) == _lib.ERR_INVALID_ARG
        assert call_list([desc(0, d_in=0)], ksize=ksize, sx=sx, t1=math.inf) == _lib.ERR_INVALID_ARG
        assert call_list([desc(0, d_in=0)], ksize=ksize, sx=sx) == _lib.ERR_INVALID_ARG


@pytest.mark.parametrize("aperture", [3, 5, 7])
def test_good_arguments_reach_the_device(aperture):
    no_gpu()
    blurs = [((5, 5), 0.0, 0.0), ((1, 1), 0.0, 0.0), ((0, 0), 1.4, 0.0), ((0, 0), 5.0, 0.0), ((31, 3), 0.0, 0.0),
             ((3, 31), 2.0, 0.5), ((5, 5), -1.0, 0.0), ((0, 9), 1.0, 1.4), ((7, 7), 0.0, -2.0)]
    for ksize, sx, sy in blurs:
        for kw in ({}, dict(ch=3), dict(h=1, w=1, n=1), dict(h=1, w=300), dict(h=300, w=1), dict(in_pitch=21, out_pitch=19), dict(l2=1)):
            assert call(ksize=ksize, sx=sx, sy=sy, aperture=aperture, **kw) == _lib.ERR_NO_DEVICE, (ksize, kw)
        for ch in (1, 3):
            descs = [desc(0, h=1, w=1, ch=ch), desc(1, h=2, w=40, ch=ch), desc(2, h=45, w=3, ch=ch)]
            assert call_list(descs, ch, ksize, sx, sy, aperture=aperture) == _lib.ERR_NO_DEVICE, (ksize, ch)


def test_ctypes_entries_and_python_wrappers():
    for name in ("b200_cv_gaussian_canny_device_strided", "b200_cv_gaussian_canny_frames_device", "b200_cv_gaussian_kernel"):
        assert name in _lib.SIGNATURES
    assert _lib.load().b200_version() == 1
    import inspect
    for fn in (cb.torch_api.cv_canny, cb.torch_api.cv_canny_color, cb.torch_api.cv_canny_list, cb.torch_api.cv_canny_color_list):
        p = inspect.signature(fn).parameters["gaussian"]
        assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is None


def test_python_wrappers_raise_c_errors():
    with pytest.raises(_lib.CannyB200Error, match="odd"):
        cb.cv_gaussian_canny_device_strided_ptr(None, IN, 16, 128, 2, 8, 16, 1, (4, 4), 0.0, 0.0, 20, 60, 3, False, OUT, 16, 128)
    with pytest.raises(_lib.CannyB200Error, match="31"):
        cb.cv_gaussian_canny_frames_device_ptr(None, [desc(0)], 1, (33, 33), 0.0, 0.0, 20, 60, 3, True)


def test_gaussian_keyword_parsing():
    from canny_edge_b200.torch_api import gaussian_args
    assert gaussian_args(None) is None
    assert gaussian_args(((5, 5), 0)) == ((5, 5), 0.0, 0.0)
    assert gaussian_args((5, 1.5)) == ((5, 5), 1.5, 0.0)
    assert gaussian_args(((9, 3), 1.5, 0.7)) == ((9, 3), 1.5, 0.7)
    assert gaussian_args([[0, 0], 2]) == ((0, 0), 2.0, 0.0)
    assert gaussian_args((np.int64(7), np.float32(0.5))) == ((7, 7), 0.5, 0.0)
    # values cv2 rejects are the library's to refuse: they parse
    assert gaussian_args(((4, 4), 0)) == ((4, 4), 0.0, 0.0)
    assert gaussian_args((5, math.nan))[1] != gaussian_args((5, math.nan))[1]
    for bad in (5, "5", (5,), (5, 1, 1, 1), ((5, 5, 5), 0), ((5.0, 5), 0), (5.0, 0), ("5", 0), ((5, 5), "0"), ((5, 5), None),
                (True, 0), ((5, 5), 0, False), {"ksize": 5}):
        with pytest.raises(ValueError):
            gaussian_args(bad)


def test_torch_front_end_rejections_on_cpu_tensors():
    import torch
    api = cb.torch_api
    x = torch.zeros((2, 32, 48), dtype=torch.uint8)
    c = torch.zeros((32, 48, 3), dtype=torch.uint8)
    for g in (((5, 5), 0), (3, 1.0, 2.0), ((1, 1), 0)):
        with pytest.raises(ValueError, match="CUDA"):
            api.cv_canny(x, 20, 60, gaussian=g)
        with pytest.raises(ValueError, match="CUDA"):
            api.cv_canny_color(c, 20, 60, gaussian=g, L2gradient=True)
        with pytest.raises(ValueError, match="CUDA"):
            api.cv_canny_list([x[0], x[1, :5, :7]], 20, 60, gaussian=g)
        with pytest.raises(ValueError, match="CUDA"):
            api.cv_canny_color_list([c], 20, 60, gaussian=g, apertureSize=5)
    for bad in ((5,), "5", ((5, 5, 5), 0)):
        for fn, arg in ((api.cv_canny, x), (api.cv_canny_color, c), (api.cv_canny_list, [x[0]]), (api.cv_canny_color_list, [c])):
            with pytest.raises(ValueError, match="gaussian"):
                fn(arg, 20, 60, gaussian=bad)
    with pytest.raises(TypeError):
        api.cv_canny(x, 20, 60, 3, False, ((5, 5), 0))   # keyword-only
