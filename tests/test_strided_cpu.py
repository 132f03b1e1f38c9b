"""CPU tests of the strided device batch: argument validation of the C entry points (it runs before any device work) and the
torch front end's stride derivation and rejections on CPU tensors."""
import ctypes as C

import numpy as np
import pytest

import canny_edge_b200 as cb
from canny_edge_b200 import _lib
from canny_edge_b200.torch_api import frame_layout

IN, OUT = 1 << 32, 1 << 40   # device addresses far apart; never dereferenced by the checks


def call(bgr, d_in=IN, in_pitch=None, in_fs=None, n=2, h=8, w=16, lo=20, hi=60, d_out=OUT, out_pitch=None, out_fs=None):
    lib = _lib.load()
    bpp = 3 if bgr else 1
    in_pitch = bpp * w if in_pitch is None else in_pitch
    in_fs = h * in_pitch if in_fs is None else in_fs
    out_pitch = w if out_pitch is None else out_pitch
    out_fs = h * out_pitch if out_fs is None else out_fs
    fn = lib.b200_canny_batch_device_bgr_strided if bgr else lib.b200_canny_batch_device_strided
    return fn(None, d_in, in_pitch, in_fs, n, h, w, C.c_float(1.4), lo, hi, d_out, out_pitch, out_fs)


@pytest.mark.parametrize("bgr", [False, True])
def test_strided_entry_points_reject_bad_layouts(bgr):
    bpp = 3 if bgr else 1
    h, w = 8, 16
    bad = {
        "null input": dict(d_in=None),
        "null output": dict(d_out=None),
        "height < 2": dict(h=1),
        "no frames": dict(n=0),
        "negative input pitch": dict(in_pitch=-bpp * w),
        "negative input frame stride": dict(in_fs=-1),
        "negative output pitch": dict(out_pitch=-w),
        "negative output frame stride": dict(out_fs=-1),
        "input pitch below a row": dict(in_pitch=bpp * w - 1),
        "output pitch below a row": dict(out_pitch=w - 1),
        "input frames overlap": dict(in_fs=(h - 1) * bpp * w + bpp * w - 1),
        "output frames overlap": dict(out_fs=(h - 1) * w + w - 1),
        "broadcast input frames": dict(in_fs=0),
        "output inside the input": dict(d_out=IN + bpp * w),
        "input inside the output": dict(d_in=OUT + w),
    }
    for name, kw in bad.items():
        assert call(bgr, **kw) == _lib.ERR_INVALID_ARG, name
        assert _lib.load().b200_last_error(), name


@pytest.mark.parametrize("bgr", [False, True])
def test_strided_entry_points_accept_good_layouts(bgr):
    """Valid layouts pass every check and stop only at the missing device (B200_ERR_NO_DEVICE here, work on a GPU box)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: these fake addresses would be used")
    bpp = 3 if bgr else 1
    h, w = 8, 16
    good = [
        {},
        dict(in_pitch=bpp * w + 5, out_pitch=w + 3),                         # odd pitches
        dict(in_fs=(h - 1) * bpp * w + bpp * w, out_fs=(h - 1) * w + w),     # frames packed as tightly as they can be
        dict(n=1, in_fs=0, out_fs=0),                                        # a single frame's stride is not used
        dict(d_out=IN + 2 * h * bpp * w),                                    # output right behind the input
        dict(lo=300, hi=400),                                                # thresholds: checked as before
    ]
    for kw in good:
        assert call(bgr, **kw) == _lib.ERR_NO_DEVICE, kw


def test_strides_that_would_overflow_are_rejected():
    """Products of huge strides are checked without wrapping: such layouts are invalid, never accepted."""
    big = (1 << 62) + 5
    for kw in (dict(in_pitch=big), dict(out_pitch=big), dict(in_fs=big), dict(out_fs=big), dict(n=1 << 30, in_fs=1 << 40),
               dict(in_pitch=1 << 45, in_fs=1 << 50)):
        assert call(False, **kw) == _lib.ERR_INVALID_ARG, kw
        assert call(True, **kw) == _lib.ERR_INVALID_ARG, kw


def test_frame_layout_of_views():
    import torch
    x = torch.zeros((5, 100, 160), dtype=torch.uint8)
    assert frame_layout(x) == (5, 100, 160, 160, 16000)
    assert frame_layout(x[0]) == (1, 100, 160, 160, 16000)
    crop = x[1:4, 10:90, 3:131]                       # unaligned column offset, pitch stays the parent's
    assert frame_layout(crop) == (3, 80, 128, 160, 16000)
    assert crop.data_ptr() - x.data_ptr() == 16000 + 10 * 160 + 3
    padded = torch.zeros((4, 64, 656), dtype=torch.uint8)[:, :, :641]
    assert frame_layout(padded) == (4, 64, 641, 656, 64 * 656)
    nchw = torch.zeros((3, 2, 50, 70), dtype=torch.uint8)
    assert frame_layout(nchw[:, 1]) == (3, 50, 70, 70, 2 * 50 * 70)
    one = x[2:3, 5:50, 7:90]                          # N == 1: the frame stride is that of a dense frame of this pitch
    assert frame_layout(one) == (1, 45, 83, 160, 45 * 160)
    bgr = torch.zeros((2, 40, 64, 3), dtype=torch.uint8)
    assert frame_layout(bgr, bgr=True) == (2, 40, 64, 192, 40 * 192)
    assert frame_layout(bgr[:, 3:30, 5:50], bgr=True) == (2, 27, 45, 192, 40 * 192)
    assert frame_layout(bgr[1], bgr=True) == (1, 40, 64, 192, 40 * 192)
    # a gray image of width 3 is gray input, not one B,G,R row
    assert frame_layout(torch.zeros((10, 3), dtype=torch.uint8)) == (1, 10, 3, 3, 30)


def test_frame_layout_rejects_what_the_kernels_cannot_address():
    import torch
    x = torch.zeros((4, 32, 48), dtype=torch.uint8)
    cases = [
        x.transpose(1, 2),                                        # columns are not unit-stride
        x[:, :, ::2],                                             # every other column
        x[0:1].expand(4, 32, 48),                                 # broadcast frames: frame stride 0
        x[:, 0:1].expand(4, 32, 48),                              # broadcast rows: row stride 0
        torch.zeros((32, 48, 3), dtype=torch.uint8).permute(2, 0, 1),   # planar channels seen as frames: not unit-stride rows
    ]
    for t in cases:
        with pytest.raises(ValueError, match=r"\.contiguous\(\)"):
            frame_layout(t)
    planar = torch.zeros((2, 3, 32, 48), dtype=torch.uint8).permute(0, 2, 3, 1)   # NCHW seen as NHWC: pixels not 3 bytes
    with pytest.raises(ValueError, match=r"\.contiguous\(\)"):
        frame_layout(planar, bgr=True)
    for t, kw in ((x.float(), {}), (x[0, 0], {}), (x[..., None], {}), (torch.zeros((1, 2), dtype=torch.uint8), {}),
                  (x, dict(bgr=True)), (torch.zeros((4, 32, 48, 4), dtype=torch.uint8), dict(bgr=True))):
        with pytest.raises(ValueError):
            frame_layout(t, **kw)
    with pytest.raises(TypeError):
        frame_layout(np.zeros((4, 4), np.uint8))


def test_torch_front_end_needs_cuda_tensors():
    import torch
    x = torch.zeros((2, 32, 48), dtype=torch.uint8)
    with pytest.raises(ValueError, match="CUDA"):
        cb.torch_api.canny(x, 1.4, 20, 60)
    with pytest.raises(ValueError, match="CUDA"):
        cb.torch_api.canny_bgr(torch.zeros((32, 48, 3), dtype=torch.uint8), 1.4, 20, 60)
    # layout errors come first, before anything touches a device
    with pytest.raises(ValueError, match=r"\.contiguous\(\)"):
        cb.torch_api.canny(x.transpose(1, 2), 1.4, 20, 60)
