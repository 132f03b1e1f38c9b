"""CPU tests of ragged frame lists (b200_canny_frames_device): argument validation runs before any device work, so every bad list
returns B200_ERR_INVALID_ARG here rather than B200_ERR_NO_DEVICE; and the torch list front end's rejections on CPU tensors."""
import ctypes as C

import pytest

import canny_edge_b200 as cb
from canny_edge_b200 import _lib
from canny_edge_b200.api import frame_list

IN, OUT = 1 << 32, 1 << 40   # device addresses far apart; never dereferenced by the checks
MB = 1 << 20


def desc(i, h=8, w=16, bgr=False, in_pitch=None, out_pitch=None, d_in=None, d_out=None):
    """Frame i of a list: inputs and outputs each 1 MB apart, so frames never overlap unless a case says so."""
    bpp = 3 if bgr else 1
    return (IN + i * MB if d_in is None else d_in, bpp * w if in_pitch is None else in_pitch,
            OUT + i * MB if d_out is None else d_out, w if out_pitch is None else out_pitch, h, w)


def call(descs, bgr=False, lo=20, hi=60, n=None):
    lib = _lib.load()
    fn = lib.b200_canny_frames_device_bgr if bgr else lib.b200_canny_frames_device
    return fn(None, frame_list(descs), len(descs) if n is None else n, C.c_float(1.4), lo, hi)


def no_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: these fake addresses would be used")


@pytest.mark.parametrize("bgr", [False, True])
def test_frames_entry_points_reject_bad_lists(bgr):
    bpp = 3 if bgr else 1
    bad = {
        "null input": [desc(0, bgr=bgr), desc(1, bgr=bgr, d_in=0)],
        "null output": [desc(0, bgr=bgr, d_out=0)],
        "height < 2": [desc(0, bgr=bgr), desc(1, h=1, bgr=bgr)],
        "width < 2": [desc(0, w=1, bgr=bgr)],
        "2 x 1": [desc(0, h=2, w=1, bgr=bgr)],
        "negative input pitch": [desc(0, bgr=bgr, in_pitch=-bpp * 16)],
        "negative output pitch": [desc(0, bgr=bgr, out_pitch=-16)],
        "input pitch below a row": [desc(0, bgr=bgr, in_pitch=bpp * 16 - 1)],
        "output pitch below a row": [desc(0, bgr=bgr, out_pitch=15)],
        "input extent above 2^48": [desc(0, bgr=bgr, in_pitch=1 << 46)],
        "output extent above 2^48": [desc(0, bgr=bgr, out_pitch=1 << 46)],
        "output/output overlap": [desc(0, bgr=bgr), desc(1, bgr=bgr, d_out=OUT + 7 * 16 + 15)],
        "output/output identical": [desc(0, bgr=bgr), desc(1, bgr=bgr, d_out=OUT)],
        "output inside an input": [desc(0, bgr=bgr, d_out=IN + bpp * 16)],
        "input inside an output": [desc(0, bgr=bgr, d_in=OUT + 16)],
        "output over another frame's input": [desc(0, bgr=bgr), desc(1, bgr=bgr, d_out=IN + 3)],
        # tiles side by side in the same rows: their extents (first to last byte) interleave
        "mosaic tiles sharing rows": [desc(0, h=8, w=16, out_pitch=64, bgr=bgr), desc(1, h=8, w=16, out_pitch=64, d_out=OUT + 16, bgr=bgr)],
    }
    for name, descs in bad.items():
        assert call(descs, bgr) == _lib.ERR_INVALID_ARG, name
        assert _lib.load().b200_last_error(), name
    assert _lib.load().b200_canny_frames_device(None, None, 1, C.c_float(1.4), 20, 60) == _lib.ERR_INVALID_ARG
    for n in (0, -1):
        assert call([desc(0, bgr=bgr)], bgr, n=n) == _lib.ERR_INVALID_ARG, n


@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_overlaps_in_long_lists(where):
    """1000 frames: one overlapping output (with another output, or with an input) is found wherever it sits in the list."""
    k = {"first": 0, "middle": 500, "last": 999}[where]
    base = [desc(i) for i in range(1000)]
    oo = list(base)
    other = 999 - k if k != 500 else 3
    oo[k] = desc(k, d_out=OUT + other * MB + 5)            # inside frame `other`'s output
    assert call(oo) == _lib.ERR_INVALID_ARG
    oi = list(base)
    oi[k] = desc(k, d_out=IN + other * MB + 100)           # inside frame `other`'s input
    assert call(oi) == _lib.ERR_INVALID_ARG
    tail = list(base)
    tail[k] = desc(k, d_out=OUT + other * MB - 10)         # its last row runs into frame `other`'s first bytes
    assert call(tail) == _lib.ERR_INVALID_ARG


def test_overflowing_pitches_are_rejected():
    big = (1 << 62) + 5
    for kw in (dict(in_pitch=big), dict(out_pitch=big), dict(in_pitch=(1 << 63) - 1), dict(out_pitch=(1 << 63) - 1),
               dict(h=1 << 20, in_pitch=1 << 29)):
        for bgr in (False, True):
            assert call([desc(0, bgr=bgr), desc(1, bgr=bgr, **kw)], bgr) == _lib.ERR_INVALID_ARG, kw


def test_unsupported_frames_and_thresholds():
    # 2^31 pixels: beyond the kernels' int indexing
    assert call([desc(0), desc(1, h=1 << 16, w=1 << 15, d_out=OUT + (1 << 33))]) == _lib.ERR_UNSUPPORTED
    assert call([desc(0)], lo=300, hi=100) == _lib.ERR_UNSUPPORTED


@pytest.mark.parametrize("bgr", [False, True])
def test_good_lists_reach_the_device(bgr):
    """Valid lists pass every check and stop only at the missing device."""
    no_gpu()
    bpp = 3 if bgr else 1
    good = {
        "one frame": [desc(0, bgr=bgr)],
        "mixed sizes": [desc(i, h=2 + i, w=2 + 3 * i, bgr=bgr) for i in range(20)],
        "duplicate input": [desc(0, bgr=bgr), desc(1, bgr=bgr, d_in=IN)],
        "overlapping inputs": [desc(0, bgr=bgr), desc(1, bgr=bgr, d_in=IN + 5)],
        "outputs back to back": [desc(0, bgr=bgr), desc(1, bgr=bgr, d_out=OUT + 7 * 16 + 16)],
        # tiles of one 64-byte-pitch mosaic in rows of their own, at any column
        "mosaic tiles": [desc(0, h=8, w=16, out_pitch=64, bgr=bgr), desc(1, h=8, w=16, out_pitch=64, d_out=OUT + 8 * 64 + 16, bgr=bgr),
                         desc(2, h=4, w=32, out_pitch=64, d_out=OUT + 16 * 64 + 32, bgr=bgr)],
        "odd pitches": [desc(0, bgr=bgr, in_pitch=bpp * 16 + 5, out_pitch=19)],
        "output right behind the input": [desc(0, bgr=bgr, d_out=IN + 8 * bpp * 16)],
        "1000 frames": [desc(i, bgr=bgr) for i in range(1000)],
    }
    for name, descs in good.items():
        assert call(descs, bgr) == _lib.ERR_NO_DEVICE, name
    assert call([desc(0, bgr=bgr)], bgr, lo=0, hi=300) == _lib.ERR_NO_DEVICE


def test_torch_list_rejections():
    import torch
    from canny_edge_b200 import torch_api
    a = torch.zeros((32, 48), dtype=torch.uint8)
    b = torch.zeros((20, 30), dtype=torch.uint8)
    with pytest.raises(ValueError, match="empty"):
        torch_api.canny_list([], 1.4, 20, 60)
    with pytest.raises(ValueError, match="CUDA"):
        torch_api.canny_list([a, b], 1.4, 20, 60)
    with pytest.raises(ValueError, match="CUDA"):
        torch_api.canny_bgr_list([torch.zeros((20, 30, 3), dtype=torch.uint8)], 1.4, 20, 60)
    with pytest.raises(ValueError, match="uint8"):
        torch_api.canny_list([a, b.float()], 1.4, 20, 60)
    with pytest.raises(ValueError, match=r"\.contiguous\(\)"):
        torch_api.canny_list([a, b.t()], 1.4, 20, 60)
    with pytest.raises(ValueError, match="expected one"):
        torch_api.canny_list([a, torch.zeros((2, 20, 30), dtype=torch.uint8)], 1.4, 20, 60)
    with pytest.raises(ValueError, match="expected one"):
        torch_api.canny_bgr_list([a], 1.4, 20, 60)
    with pytest.raises(ValueError, match="2 tensors for 1"):
        torch_api.canny_list([a], 1.4, 20, 60, out=[a.clone(), a.clone()])
    with pytest.raises(ValueError, match="shape"):
        torch_api.canny_list([a, b], 1.4, 20, 60, out=[a.clone(), a.clone()])
    with pytest.raises(TypeError):
        torch_api.canny_list([a, b.numpy()], 1.4, 20, 60)
