"""CPU tests of OpenCV-compatible frame lists (b200_cv_canny_frames_device): the channel, threshold and list checks all run before any
device work, in that order, so every bad call returns its error here rather than B200_ERR_NO_DEVICE; and the torch list front end's
rejections (torch_api.cv_canny_list / cv_canny_color_list) on CPU tensors."""
import ctypes as C
import math

import pytest

import canny_edge_b200 as cb
from canny_edge_b200 import _lib
from canny_edge_b200.api import frame_list

IN, OUT = 1 << 32, 1 << 40   # device addresses far apart; never dereferenced by the checks
MB = 1 << 20


def desc(i, h=8, w=16, ch=1, in_pitch=None, out_pitch=None, d_in=None, d_out=None):
    """Frame i of a list: inputs and outputs each 1 MB apart, so frames never overlap unless a case says so."""
    return (IN + i * MB if d_in is None else d_in, ch * w if in_pitch is None else in_pitch,
            OUT + i * MB if d_out is None else d_out, w if out_pitch is None else out_pitch, h, w)


def call(descs, ch=1, t1=20.0, t2=60.0, l2=0, n=None, channels=None):
    lib = _lib.load()
    return lib.b200_cv_canny_frames_device(None, frame_list(descs), len(descs) if n is None else n, ch if channels is None else channels,
                                           C.c_double(t1), C.c_double(t2), l2)


def no_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: these fake addresses would be used")


@pytest.mark.parametrize("ch", [1, 3])
def test_bad_lists_are_rejected(ch):
    bad = {
        "null input": [desc(0, ch=ch), desc(1, ch=ch, d_in=0)],
        "null output": [desc(0, ch=ch, d_out=0)],
        "height 0": [desc(0, ch=ch), desc(1, h=0, ch=ch)],
        "width 0": [desc(0, w=0, ch=ch)],
        "negative height": [desc(0, h=-3, ch=ch)],
        "negative input pitch": [desc(0, ch=ch, in_pitch=-ch * 16)],
        "negative output pitch": [desc(0, ch=ch, out_pitch=-16)],
        "input pitch below a row": [desc(0, ch=ch, in_pitch=ch * 16 - 1)],
        "output pitch below a row": [desc(0, ch=ch, out_pitch=15)],
        "input extent above 2^48": [desc(0, ch=ch, in_pitch=1 << 46)],
        "output extent above 2^48": [desc(0, ch=ch, out_pitch=1 << 46)],
        "output/output overlap": [desc(0, ch=ch), desc(1, ch=ch, d_out=OUT + 7 * 16 + 15)],
        "output/output identical": [desc(0, ch=ch), desc(1, ch=ch, d_out=OUT)],
        "output inside an input": [desc(0, ch=ch, d_out=IN + ch * 16)],
        "input inside an output": [desc(0, ch=ch, d_in=OUT + 16)],
        "output over another frame's input": [desc(0, ch=ch), desc(1, ch=ch, d_out=IN + 3)],
        "1x1 outputs on one byte": [desc(0, h=1, w=1, ch=ch), desc(1, h=1, w=1, ch=ch, d_out=OUT)],
        # tiles side by side in the same rows: their extents (first to last byte) interleave
        "mosaic tiles sharing rows": [desc(0, h=8, w=16, out_pitch=64, ch=ch), desc(1, h=8, w=16, out_pitch=64, d_out=OUT + 16, ch=ch)],
    }
    for name, descs in bad.items():
        assert call(descs, ch) == _lib.ERR_INVALID_ARG, name
        assert _lib.load().b200_last_error(), name
    lib = _lib.load()
    assert lib.b200_cv_canny_frames_device(None, None, 1, ch, C.c_double(20), C.c_double(60), 0) == _lib.ERR_INVALID_ARG
    for n in (0, -1):
        assert call([desc(0, ch=ch)], ch, n=n) == _lib.ERR_INVALID_ARG, n


def test_gray_pitch_is_too_small_for_three_channels():
    """A pitch of one byte per pixel is a full gray row and a third of a 3-channel row."""
    assert call([desc(0, ch=1, in_pitch=16)], 3) == _lib.ERR_INVALID_ARG
    assert call([desc(0, ch=1, in_pitch=47)], 3) == _lib.ERR_INVALID_ARG


@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_overlaps_in_long_lists(where):
    """1000 frames: one overlapping output (with another output, or with an input) is found wherever it sits in the list."""
    k = {"first": 0, "middle": 500, "last": 999}[where]
    other = 999 - k if k != 500 else 3
    for ch in (1, 3):
        base = [desc(i, ch=ch) for i in range(1000)]
        for d_out in (OUT + other * MB + 5, IN + other * MB + 100, OUT + other * MB - 10):
            lst = list(base)
            lst[k] = desc(k, ch=ch, d_out=d_out)
            assert call(lst, ch) == _lib.ERR_INVALID_ARG, (ch, d_out)


def test_overflowing_pitches_are_rejected():
    big = (1 << 62) + 5
    for kw in (dict(in_pitch=big), dict(out_pitch=big), dict(in_pitch=(1 << 63) - 1), dict(out_pitch=(1 << 63) - 1),
               dict(h=1 << 20, in_pitch=1 << 29)):
        for ch in (1, 3):
            assert call([desc(0, ch=ch), desc(1, ch=ch, **kw)], ch) == _lib.ERR_INVALID_ARG, kw


@pytest.mark.parametrize("channels", [0, 2, 4, -1, 255])
def test_channel_counts_are_unsupported(channels):
    """Checked first: even a list that is bad in every other way returns UNSUPPORTED for the channel count."""
    assert call([desc(0)], channels=channels) == _lib.ERR_UNSUPPORTED
    assert call([desc(0, d_in=0)], channels=channels, t1=math.nan) == _lib.ERR_UNSUPPORTED
    assert _lib.load().b200_cv_canny_frames_device(None, None, 0, channels, C.c_double(20), C.c_double(60), 0) == _lib.ERR_UNSUPPORTED


@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("l2", [0, 1])
def test_thresholds_are_checked_before_the_list(ch, l2):
    inf = math.inf
    for t1, t2 in ((math.nan, 60), (20, math.nan), (inf, 60), (20, -inf), (math.nan, math.nan)):
        assert call([desc(0, ch=ch)], ch, t1, t2, l2) == _lib.ERR_INVALID_ARG, (t1, t2)
        assert call([desc(0, ch=ch, d_out=0)], ch, t1, t2, l2) == _lib.ERR_INVALID_ARG, (t1, t2)
    # floors outside int32 (for L2 after clamping to 32767 and squaring, which stays inside): refused, never computed wrongly
    big = [(1e10, 20), (20, 2.0 ** 31), (-(2.0 ** 31) - 1, 20), (-1e12, 1e12)] if not l2 else [(-(2.0 ** 31) - 1, 20), (-1e12, 5)]
    for t1, t2 in big:
        assert call([desc(0, ch=ch)], ch, t1, t2, l2) == _lib.ERR_UNSUPPORTED, (t1, t2)
        # the threshold check comes before the list checks: a bad list does not hide it
        assert call([desc(0, ch=ch, d_in=0)], ch, t1, t2, l2) == _lib.ERR_UNSUPPORTED, (t1, t2)


def test_unsupported_frames():
    # 2^31 pixels: beyond the kernels' int indexing
    for ch in (1, 3):
        assert call([desc(0, ch=ch), desc(1, h=1 << 16, w=1 << 15, ch=ch, d_out=OUT + (1 << 33), d_in=IN + (1 << 33))], ch) \
            == _lib.ERR_UNSUPPORTED


@pytest.mark.parametrize("ch", [1, 3])
def test_good_lists_reach_the_device(ch):
    """Valid lists pass every check and stop only at the missing device."""
    no_gpu()
    good = {
        "one frame": [desc(0, ch=ch)],
        "1x1": [desc(0, h=1, w=1, ch=ch)],
        "1xN and Nx1": [desc(0, h=1, w=37, ch=ch), desc(1, h=45, w=1, ch=ch), desc(2, h=1, w=1, ch=ch)],
        "mixed sizes": [desc(i, h=1 + i, w=1 + 3 * i, ch=ch) for i in range(20)],
        "duplicate input": [desc(0, ch=ch), desc(1, ch=ch, d_in=IN)],
        "overlapping inputs": [desc(0, ch=ch), desc(1, ch=ch, d_in=IN + 5)],
        "outputs back to back": [desc(0, ch=ch), desc(1, ch=ch, d_out=OUT + 7 * 16 + 16)],
        "1x1 outputs back to back": [desc(0, h=1, w=1, ch=ch), desc(1, h=1, w=1, ch=ch, d_out=OUT + 1)],
        # tiles of one 64-byte-pitch mosaic in rows of their own, at any column
        "mosaic tiles": [desc(0, h=8, w=16, out_pitch=64, ch=ch), desc(1, h=8, w=16, out_pitch=64, d_out=OUT + 8 * 64 + 16, ch=ch),
                         desc(2, h=4, w=32, out_pitch=64, d_out=OUT + 16 * 64 + 32, ch=ch)],
        "odd pitches": [desc(0, ch=ch, in_pitch=ch * 16 + 5, out_pitch=19)],
        "output right behind the input": [desc(0, ch=ch, d_out=IN + 8 * ch * 16)],
        # taller than the uniform call's 65535 x 64 rows: the list's grid is 1-D
        "very tall frame": [desc(0, h=5_000_000, w=1, ch=ch, in_pitch=ch)],
        "1000 frames": [desc(i, ch=ch) for i in range(1000)],
    }
    for name, descs in good.items():
        assert call(descs, ch) == _lib.ERR_NO_DEVICE, name
    for t1, t2, l2 in ((60, 20, 0), (-5, -1, 0), (0, 0, 1), (1e9, 1e9, 1), (2.0 ** 31 - 1, 0, 0), (-(2.0 ** 31), 5, 0)):
        assert call([desc(0, ch=ch)], ch, t1, t2, l2) == _lib.ERR_NO_DEVICE, (t1, t2, l2)


def test_ctypes_entry_and_python_wrapper_exist():
    assert "b200_cv_canny_frames_device" in _lib.SIGNATURES
    assert callable(cb.cv_canny_frames_device_ptr)
    with pytest.raises(cb.CannyB200Error) as e:
        cb.cv_canny_frames_device_ptr(None, [desc(0)], 2, 20, 60, False)
    assert e.value.status == _lib.ERR_UNSUPPORTED


@pytest.mark.parametrize("color", [False, True])
def test_torch_list_rejections(color):
    import torch
    from canny_edge_b200 import torch_api
    fn = torch_api.cv_canny_color_list if color else torch_api.cv_canny_list
    shape = (lambda h, w: (h, w, 3)) if color else (lambda h, w: (h, w))
    a = torch.zeros(shape(32, 48), dtype=torch.uint8)
    b = torch.zeros(shape(20, 30), dtype=torch.uint8)
    one = torch.zeros(shape(1, 1), dtype=torch.uint8)
    with pytest.raises(ValueError, match="empty"):
        fn([], 20, 60)
    with pytest.raises(ValueError, match="CUDA"):          # CPU tensors, 1 x 1 frames included
        fn([a, b, one], 20, 60)
    with pytest.raises(ValueError, match="CUDA"):
        fn([a], 20, 60, L2gradient=True)
    with pytest.raises(ValueError, match="uint8"):
        fn([a, b.float()], 20, 60)
    with pytest.raises(ValueError, match="expected one"):  # wrong dims
        fn([a, torch.zeros((2,) + shape(20, 30), dtype=torch.uint8)], 20, 60)
    with pytest.raises(ValueError, match="expected one"):
        fn([torch.zeros(shape(20, 30)[:-1] if color else (20, 30, 3), dtype=torch.uint8)], 20, 60)
    with pytest.raises(ValueError, match="at least 1 x 1"):
        fn([torch.zeros(shape(0, 5), dtype=torch.uint8)], 20, 60)
    with pytest.raises(ValueError, match="2 tensors for 1"):
        fn([a], 20, 60, out=[torch.zeros((32, 48), dtype=torch.uint8)] * 2)
    with pytest.raises(ValueError, match="shape"):
        fn([a, b], 20, 60, out=[torch.zeros((32, 48), dtype=torch.uint8)] * 2)
    with pytest.raises(ValueError, match="shape"):
        fn([a], 20, 60, out=[torch.zeros(shape(32, 48), dtype=torch.uint8)] if color else [torch.zeros((48, 32), dtype=torch.uint8)])
    with pytest.raises(TypeError):
        fn([a, b.numpy()], 20, 60)


def test_torch_list_rejects_rows_that_are_not_contiguous():
    import torch
    from canny_edge_b200 import torch_api
    g = torch.zeros((20, 30), dtype=torch.uint8)
    with pytest.raises(ValueError, match=r"\.contiguous\(\)"):
        torch_api.cv_canny_list([g, g.t()], 20, 60)
    with pytest.raises(ValueError, match=r"\.contiguous\(\)"):
        torch_api.cv_canny_list([g[:, ::2]], 20, 60)
    c = torch.zeros((20, 30, 3), dtype=torch.uint8)
    with pytest.raises(ValueError, match=r"\.contiguous\(\)"):
        torch_api.cv_canny_color_list([torch.zeros((3, 20, 30), dtype=torch.uint8).permute(1, 2, 0)], 20, 60)   # planar
    with pytest.raises(ValueError, match=r"\.contiguous\(\)"):
        torch_api.cv_canny_color_list([c[:, ::2]], 20, 60)


def test_torch_list_rejects_mixed_devices():
    """A list whose tensors are not all on one CUDA device is refused before any call; on a CPU-only machine the first non-CUDA
    tensor is what is reported."""
    import torch
    from canny_edge_b200 import torch_api
    g = torch.zeros((20, 30), dtype=torch.uint8)
    if torch.cuda.is_available():
        with pytest.raises(ValueError, match="one device|CUDA"):
            torch_api.cv_canny_list([g.cuda(), g], 20, 60)
        with pytest.raises(ValueError, match="CUDA"):
            torch_api.cv_canny_list([g.cuda()], 20, 60, out=[torch.zeros((20, 30), dtype=torch.uint8)])
    else:
        meta = torch.zeros((20, 30), dtype=torch.uint8, device="meta")
        with pytest.raises(ValueError, match="CUDA"):
            torch_api.cv_canny_list([meta, g], 20, 60)
        with pytest.raises(ValueError, match="CUDA"):
            torch_api.cv_canny_list([g], 20, 60, out=[meta])
