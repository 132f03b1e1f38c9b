"""The OpenCV-compatible path on the B200 (torch_api.cv_canny / cv_canny_color, b200_cv_canny_device_strided): every map against the
numpy restatement of cv::Canny (oracle/cv_canny.py) bit for bit, and against cv2.Canny where cv2 is importable.  Outputs sit in
sentinel-filled buffers whose padding must survive."""
import numpy as np
import pytest

import canny_edge_b200 as cb
from oracle.cv_canny import cv_canny

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5

try:
    import cv2
except Exception:   # cv2 is optional: the restatement is the specification
    cv2 = None


@pytest.fixture(scope="module")
def ctx():
    c = cb.Context(0)
    yield c
    c.close()


def want_map(img, lo, hi, l2):
    want = cv_canny(img, lo, hi, l2)
    if cv2 is not None:
        assert np.array_equal(want, cv2.Canny(np.ascontiguousarray(img), lo, hi, L2gradient=l2)), "restatement != cv2.Canny"
    return want


def content(kind, n, h, w, ch, seed):
    """(n, h, w) or (n, h, w, ch) uint8 frames: shapes, noise (every pixel a candidate at low thresholds), constant, ramps."""
    rng = np.random.default_rng(seed)
    if kind in ("shapes", "noise", "const"):
        k = {"shapes": 0, "noise": 1, "const": 2}[kind]
        planes = [cb.synth_host(n, h, w, kind=k, seed=seed + 17 * c) for c in range(ch)]
    else:
        planes = [rng.integers(0, 256, (n, h, w), dtype=np.uint8) // 64 * 64 for _ in range(ch)]   # blocks of 4 levels
    return planes[0] if ch == 1 else np.stack(planes, axis=-1)


def sentinel_like(n, h, w, pitch, fpad):
    import torch
    return torch.full((n, h + fpad, pitch), SENTINEL, dtype=torch.uint8, device="cuda")


def run_and_check(frames_dev, host, lo, hi, l2, out=None, ctx=None, name=""):
    """frames_dev: CUDA view of `host` ((N, H, W) or (N, H, W, 3)); out: a view into a sentinel buffer, or None."""
    import torch
    color = host.ndim == 4
    fn = cb.torch_api.cv_canny_color if color else cb.torch_api.cv_canny
    res = fn(frames_dev, lo, hi, L2gradient=l2, out=out, ctx=ctx)
    torch.cuda.synchronize()
    got = res.cpu().numpy()
    for f in range(host.shape[0]):
        want = want_map(host[f], lo, hi, l2)
        diff = int((got[f] != want).sum())
        assert diff == 0, f"{name}: frame {f} (l2={l2}, {lo}, {hi}) differs in {diff} pixels"
    return res


def check_padding(buf, n, h, w, name):
    pad = buf.cpu().numpy().copy()
    pad[:n, :h, :w] = SENTINEL
    assert (pad == SENTINEL).all(), f"{name}: bytes outside the maps were written"


@pytest.mark.parametrize("l2", [False, True])
@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("h,w", [(1, 1), (1, 37), (45, 1), (2, 2), (3, 129), (67, 131), (130, 255), (64, 128)])
def test_small_sizes(ctx, l2, ch, h, w):
    import torch
    for kind in ("shapes", "noise", "blocks"):
        host = content(kind, 2, h, w, ch, seed=h * 1000 + w)
        buf = sentinel_like(2, h, w, w + 5, 1)
        out = buf[:, :h, :w]
        run_and_check(torch.from_numpy(host).cuda(), host, 20, 60, l2, out=out, ctx=ctx, name=f"{kind} {h}x{w}x{ch}")
        check_padding(buf, 2, h, w, f"{kind} {h}x{w}x{ch}")


@pytest.mark.parametrize("l2", [False, True])
@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("h,w", [(1080, 1920), (2160, 3840)])
def test_large_frames(ctx, l2, ch, h, w):
    import torch
    host = content("shapes", 1, h, w, ch, seed=5)
    host[0, h // 3:h // 2] = np.random.default_rng(1).integers(0, 256, host[0, h // 3:h // 2].shape, dtype=np.uint8)   # a noise band
    lo, hi = (50.0, 150.0) if not l2 else (30.5, 90.0)
    run_and_check(torch.from_numpy(host).cuda(), host, lo, hi, l2, ctx=ctx, name=f"{h}x{w}x{ch}")


@pytest.mark.parametrize("l2", [False, True])
@pytest.mark.parametrize("kind", ["shapes", "noise", "const", "blocks"])
def test_contents_and_batches(ctx, l2, kind):
    import torch
    n, h, w = 5, 300, 517
    for ch in (1, 3):
        host = content(kind, n, h, w, ch, seed=11)
        for lo, hi in ((20, 60), (0, 0), (-10, 500)):
            run_and_check(torch.from_numpy(host).cuda(), host, lo, hi, l2, ctx=ctx, name=f"{kind} ch={ch}")


@pytest.mark.parametrize("l2", [False, True])
def test_test_gray(ctx, test_gray, l2):
    import torch
    host = np.ascontiguousarray(test_gray[None])
    color = np.stack([test_gray, test_gray[::-1], test_gray[:, ::-1]], axis=-1)[None]
    for lo, hi in ((20, 60), (100, 200), (60, 20), (10.5, 30.75)):
        run_and_check(torch.from_numpy(host).cuda(), host, lo, hi, l2, ctx=ctx, name="test_gray")
        run_and_check(torch.from_numpy(color).cuda(), color, lo, hi, l2, ctx=ctx, name="test_gray color")


@pytest.mark.parametrize("l2", [False, True])
def test_multi_chunk(l2):
    import torch
    c = cb.Context(0)
    try:
        c.set_chunk_frames(2)
        for ch in (1, 3):
            host = content("shapes", 7, 200, 300, ch, seed=3)
            host[1] = content("noise", 1, 200, 300, ch, seed=4)[0]
            buf = sentinel_like(7, 200, 300, 304, 2)
            out = buf[:, :200, :300]
            run_and_check(torch.from_numpy(host).cuda(), host, 20, 60, l2, out=out, ctx=c, name=f"chunks ch={ch}")
            check_padding(buf, 7, 200, 300, "chunks")
    finally:
        c.close()


@pytest.mark.parametrize("l2", [False, True])
def test_crops_pitches_and_channel_views(ctx, l2):
    import torch
    rng = np.random.default_rng(2)
    big = content("shapes", 3, 400, 700, 1, seed=8)
    big[:, 100:180] = rng.integers(0, 256, big[:, 100:180].shape, dtype=np.uint8)
    dev = torch.from_numpy(big).cuda()
    for (y0, y1, x0, x1) in ((0, 400, 0, 700), (16, 300, 16, 656), (3, 397, 5, 690), (1, 2, 7, 600), (10, 300, 699, 700)):
        host = np.ascontiguousarray(big[:, y0:y1, x0:x1])
        h, w = host.shape[1:]
        buf = sentinel_like(3, h, w, w + 7, 3)
        run_and_check(dev[:, y0:y1, x0:x1], host, 20, 60, l2, out=buf[:, :h, :w], ctx=ctx, name=f"crop {(y0, y1, x0, x1)}")
        check_padding(buf, 3, h, w, "crop")
    # one channel of an NCHW tensor
    nchw = torch.from_numpy(np.stack([big, big[:, ::-1].copy(), big[:, :, ::-1].copy()], axis=1)).cuda()
    host = np.ascontiguousarray(big[:, ::-1])
    run_and_check(nchw[:, 1], host, 20, 60, l2, ctx=ctx, name="NCHW channel")
    # (N, H, W, 3) crops, aligned and unaligned, into padded outputs
    col = content("shapes", 2, 300, 500, 3, seed=9)
    col[:, 50:90] = rng.integers(0, 256, col[:, 50:90].shape, dtype=np.uint8)
    dcol = torch.from_numpy(col).cuda()
    for (y0, y1, x0, x1) in ((0, 300, 16, 496), (7, 250, 3, 499), (1, 300, 0, 1)):
        host = np.ascontiguousarray(col[:, y0:y1, x0:x1])
        h, w = host.shape[1:3]
        buf = sentinel_like(2, h, w, w + 9, 1)
        run_and_check(dcol[:, y0:y1, x0:x1], host, 20, 60, l2, out=buf[:, :h, :w], ctx=ctx, name=f"color crop {(y0, y1, x0, x1)}")
        check_padding(buf, 2, h, w, "color crop")
    # a padded tensor whose base is 16-byte aligned and pitch a multiple of 16 (wide loads) vs odd pitch (byte loads)
    for pitch in (720, 701):
        padded = torch.zeros((3, 400, pitch), dtype=torch.uint8, device="cuda")
        padded[:, :, :700] = dev
        run_and_check(padded[:, :, :700], big, 20, 60, l2, ctx=ctx, name=f"pitch {pitch}")


@pytest.mark.parametrize("l2", [False, True])
def test_threshold_edge_cases(ctx, l2):
    import torch
    host = content("shapes", 2, 150, 260, 3, seed=21)
    host[1] = content("noise", 1, 150, 260, 3, seed=22)[0]
    dev = torch.from_numpy(host).cuda()
    for lo, hi in ((0, 0), (-1, -1), (-100.5, 0.5), (255, 256), (2040, 2040), (2039.9, 2040.1), (1e6, 1e6), (5, 1e9),
                   (32767, 40000), (1e9, 10), (0.999, 1.001), (2.0 ** 31 - 1, 0), (-(2.0 ** 31), 100)):
        run_and_check(dev, host, lo, hi, l2, ctx=ctx, name="thresholds")
    with pytest.raises(cb.CannyB200Error):   # a floor outside int32 is refused, never computed wrongly
        cb.torch_api.cv_canny_color(dev, 10, 1e10, L2gradient=False, ctx=ctx)


def test_non_default_stream(ctx):
    import torch
    host = content("shapes", 3, 260, 400, 1, seed=31)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        dev = torch.from_numpy(host).cuda(non_blocking=False)
        out = torch.empty_like(dev)
        res = cb.torch_api.cv_canny(dev, 20, 60, out=out, ctx=ctx)
        res2 = cb.torch_api.cv_canny(dev, 20, 60, L2gradient=True, ctx=ctx)
    s.synchronize()
    for f in range(3):
        assert np.array_equal(res.cpu().numpy()[f], want_map(host[f], 20, 60, False))
        assert np.array_equal(res2.cpu().numpy()[f], want_map(host[f], 20, 60, True))


def test_alternating_with_reference_semantics(ctx, oracle):
    """cv_canny and the reference's canny alternated on one context: the hysteresis switch is per launch, so the reference maps
    (with its one-way link at (1,0)/(0,1)) stay equal to the reference oracle and the OpenCV maps to cv::Canny."""
    import torch
    rng = np.random.default_rng(41)
    for i in range(6):
        n, h, w = 3, int(rng.integers(2, 300)), int(rng.integers(2, 400))
        host = content(("shapes", "noise", "blocks")[i % 3], n, h, w, 1, seed=50 + i)
        dev = torch.from_numpy(host).cuda()
        ref = cb.torch_api.canny(dev, 1.4, 20, 60, ctx=ctx)
        cvm = cb.torch_api.cv_canny(dev, 20, 60, L2gradient=bool(i & 1), ctx=ctx)
        ref2 = cb.torch_api.canny(dev, 1.0, 0, 30, ctx=ctx)
        torch.cuda.synchronize()
        for f in range(n):
            assert np.array_equal(ref.cpu().numpy()[f].astype(np.int16), oracle.canny(host[f], 1.4, 20, 60)), (i, f)
            assert np.array_equal(ref2.cpu().numpy()[f].astype(np.int16), oracle.canny(host[f], 1.0, 0, 30)), (i, f)
            assert np.array_equal(cvm.cpu().numpy()[f], want_map(host[f], 20, 60, bool(i & 1))), (i, f)


def test_seeded_fuzz(ctx):
    """120 seeded cases: sizes, channel counts, L1 / L2, layouts (dense, padded pitch, unaligned crop), contents, thresholds."""
    import torch
    rng = np.random.default_rng(20261021)
    for i in range(120):
        ch = int(rng.choice([1, 3]))
        n = int(rng.integers(1, 4))
        h, w = int(rng.integers(1, 200)), int(rng.integers(1, 300))
        l2 = bool(rng.integers(0, 2))
        kind = ("shapes", "noise", "const", "blocks")[int(rng.integers(0, 4))]
        host = content(kind, n, h, w, ch, seed=1000 + i)
        lo, hi = float(rng.uniform(-20, 300)), float(rng.uniform(-20, 600))
        if rng.integers(0, 3) == 0:
            lo, hi = float(int(lo)), float(int(hi))
        layout = int(rng.integers(0, 3))
        if layout == 0:
            dev = torch.from_numpy(host).cuda()
        else:
            ox, oy = (16, 16) if layout == 1 else (int(rng.integers(1, 16)), int(rng.integers(1, 5)))
            big = torch.zeros((n, h + oy + 2, w + ox + 5) + host.shape[3:], dtype=torch.uint8, device="cuda")
            big[:, oy:oy + h, ox:ox + w] = torch.from_numpy(host).cuda()
            dev = big[:, oy:oy + h, ox:ox + w]
        buf = sentinel_like(n, h, w, w + int(rng.integers(0, 9)), 1)
        run_and_check(dev, host, lo, hi, l2, out=buf[:, :h, :w], ctx=ctx, name=f"fuzz {i} {kind} {n}x{h}x{w}x{ch}")
        check_padding(buf, n, h, w, f"fuzz {i}")
