"""cv::Canny's apertureSize 5 and 7 on the B200 (torch_api.cv_canny / cv_canny_color / cv_canny_list / cv_canny_color_list with
apertureSize, b200_cv_canny_aperture_device_strided and b200_cv_canny_aperture_frames_device): every map against the numpy
restatement (tests/cv_canny_aperture_ref.py) bit for bit, and against cv2.Canny where cv2 is importable.  Outputs sit in
sentinel-filled buffers whose padding must survive."""
import ctypes as C

import numpy as np
import pytest

import canny_edge_b200 as cb
from canny_edge_b200 import _lib
from canny_edge_b200.api import frame_list
from cv_canny_aperture_ref import cv_canny
from test_gpu_cv_canny import SENTINEL, check_padding, content, sentinel_like
from test_gpu_cv_ragged import Outs, place

pytestmark = pytest.mark.gpu

try:
    import cv2
except Exception:   # cv2 is optional: the restatement is the specification
    cv2 = None

# thresholds that give each aperture a comparable edge density: magnitudes grow about 16x at 5 and 7 (7 after its 1/16, which
# also divides its thresholds)
SCALE = {3: 1, 5: 16, 7: 256}


def thr(a, lo=20, hi=60):
    return lo * SCALE[a], hi * SCALE[a]


def want_map(img, lo, hi, l2, a):
    want = cv_canny(img, lo, hi, l2, a)
    if cv2 is not None:
        got = cv2.Canny(np.ascontiguousarray(img), lo, hi, apertureSize=a, L2gradient=l2)
        assert np.array_equal(want, got), "restatement != cv2.Canny"
    return want


def run_and_check(frames_dev, host, lo, hi, l2, a, out=None, ctx=None, name=""):
    """frames_dev: CUDA view of `host` ((N, H, W) or (N, H, W, 3)); out: a view into a sentinel buffer, or None."""
    import torch
    fn = cb.torch_api.cv_canny_color if host.ndim == 4 else cb.torch_api.cv_canny
    res = fn(frames_dev, lo, hi, apertureSize=a, L2gradient=l2, out=out, ctx=ctx)
    torch.cuda.synchronize()
    got = res.cpu().numpy()
    for f in range(host.shape[0]):
        diff = int((got[f] != want_map(host[f], lo, hi, l2, a)).sum())
        assert diff == 0, f"{name}: frame {f} (aperture {a}, l2={l2}, {lo}, {hi}) differs in {diff} pixels"
    return res


def run_list_and_check(hosts, lo, hi, l2, a, rng, ctx=None, name="", aligned=None, outs=None):
    """hosts: (h, w) / (h, w, 3) arrays of one channel count, placed with 16-byte or byte staging; outs: views or None (then
    Outs, one sentinel buffer per map)."""
    import torch
    devs = [place(x, (i % 2 == 0) if aligned is None else aligned, rng) for i, x in enumerate(hosts)]
    sentinel = Outs([x.shape[:2] for x in hosts], rng) if outs is None else None
    views = sentinel.views if outs is None else outs
    fn = cb.torch_api.cv_canny_color_list if hosts[0].ndim == 3 else cb.torch_api.cv_canny_list
    res = fn(devs, lo, hi, apertureSize=a, L2gradient=l2, out=views, ctx=ctx)
    torch.cuda.synchronize()
    assert all(r is v for r, v in zip(res, views))
    for i, (x, r) in enumerate(zip(hosts, res)):
        diff = int((r.cpu().numpy() != want_map(x, lo, hi, l2, a)).sum())
        assert diff == 0, f"{name}: frame {i} {x.shape} (aperture {a}, l2={l2}, {lo}, {hi}) differs in {diff} pixels"
    if sentinel is not None:
        sentinel.check_padding(name)
    return res


@pytest.mark.parametrize("l2", [False, True])
@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("a", [5, 7])
def test_small_sizes_and_tile_edges(gpu_ctx, a, ch, l2):
    import torch
    sizes = [(1, 1), (1, 37), (45, 1), (2, 2), (3, 3), (5, 7), (7, 5), (63, 127), (64, 128), (65, 129), (63, 129), (65, 127),
             (130, 255)]
    for h, w in sizes:
        for kind in ("shapes", "noise", "const", "blocks"):
            host = content(kind, 2, h, w, ch, seed=h * 1000 + w)
            buf = sentinel_like(2, h, w, w + 5, 1)
            lo, hi = thr(a)
            run_and_check(torch.from_numpy(host).cuda(), host, lo, hi, l2, a, out=buf[:, :h, :w], ctx=gpu_ctx,
                          name=f"{kind} {h}x{w}x{ch}")
            check_padding(buf, 2, h, w, f"{kind} {h}x{w}x{ch}")


@pytest.mark.parametrize("l2", [False, True])
@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("a", [5, 7])
def test_large_frames(gpu_ctx, a, ch, l2):
    import torch
    for h, w in ((1080, 1920), (2160, 3840)):
        host = content("shapes", 1, h, w, ch, seed=5)
        band = host[0, h // 3:h // 2]
        host[0, h // 3:h // 2] = np.random.default_rng(1).integers(0, 256, band.shape, dtype=np.uint8)   # a noise band
        lo, hi = thr(a, 50, 150) if not l2 else thr(a, 30.5, 90)
        run_and_check(torch.from_numpy(host).cuda(), host, lo, hi, l2, a, ctx=gpu_ctx, name=f"{h}x{w}x{ch}")


@pytest.mark.parametrize("a", [5, 7])
def test_crops_pitches_and_channel_views(gpu_ctx, a):
    import torch
    rng = np.random.default_rng(2)
    lo, hi = thr(a)
    big = content("shapes", 3, 400, 700, 1, seed=8)
    big[:, 100:180] = rng.integers(0, 256, big[:, 100:180].shape, dtype=np.uint8)
    dev = torch.from_numpy(big).cuda()
    for l2 in (False, True):
        # (16, 656): base and pitch on 16-byte boundaries (16-byte staging); the others take byte loads
        for (y0, y1, x0, x1) in ((16, 300, 16, 656), (3, 397, 5, 690), (1, 2, 7, 600), (10, 300, 699, 700)):
            host = np.ascontiguousarray(big[:, y0:y1, x0:x1])
            h, w = host.shape[1:]
            buf = sentinel_like(3, h, w, w + 7, 3)
            run_and_check(dev[:, y0:y1, x0:x1], host, lo, hi, l2, a, out=buf[:, :h, :w], ctx=gpu_ctx, name=f"crop {(y0, y1, x0, x1)}")
            check_padding(buf, 3, h, w, "crop")
        nchw = torch.from_numpy(np.stack([big, big[:, ::-1].copy(), big[:, :, ::-1].copy()], axis=1)).cuda()
        run_and_check(nchw[:, 1], np.ascontiguousarray(big[:, ::-1]), lo, hi, l2, a, ctx=gpu_ctx, name="NCHW channel")
        for pitch in (720, 701):
            padded = torch.zeros((3, 400, pitch), dtype=torch.uint8, device="cuda")
            padded[:, :, :700] = dev
            run_and_check(padded[:, :, :700], big, lo, hi, l2, a, ctx=gpu_ctx, name=f"pitch {pitch}")
    col = content("shapes", 2, 300, 500, 3, seed=9)
    col[:, 50:90] = rng.integers(0, 256, col[:, 50:90].shape, dtype=np.uint8)
    dcol = torch.from_numpy(col).cuda()
    for (y0, y1, x0, x1) in ((0, 300, 16, 496), (7, 250, 3, 499), (1, 300, 0, 1)):
        host = np.ascontiguousarray(col[:, y0:y1, x0:x1])
        h, w = host.shape[1:3]
        buf = sentinel_like(2, h, w, w + 9, 1)
        run_and_check(dcol[:, y0:y1, x0:x1], host, lo, hi, True, a, out=buf[:, :h, :w], ctx=gpu_ctx, name=f"color crop {(y0, y1, x0, x1)}")
        check_padding(buf, 2, h, w, "color crop")


@pytest.mark.parametrize("a", [5, 7])
def test_multi_chunk(a):
    import torch
    c = cb.Context(0)
    try:
        c.set_chunk_frames(2)
        for ch in (1, 3):
            host = content("shapes", 7, 200, 300, ch, seed=3)
            host[1] = content("noise", 1, 200, 300, ch, seed=4)[0]
            buf = sentinel_like(7, 200, 300, 304, 2)
            run_and_check(torch.from_numpy(host).cuda(), host, *thr(a), ch == 3, a, out=buf[:, :200, :300], ctx=c,
                          name=f"chunks ch={ch}")
            check_padding(buf, 7, 200, 300, "chunks")
    finally:
        c.close()


@pytest.mark.parametrize("l2", [False, True])
@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("a", [5, 7])
def test_lists_of_mixed_sizes(gpu_ctx, a, ch, l2):
    """1x1 to 4K in one list, contents mixed, 16-byte and byte staging alternating, then byte staging only."""
    rng = np.random.default_rng(7 + ch + 10 * l2 + a)
    sizes = [(1, 1), (2160, 3840), (1, 37), (45, 1), (256, 256), (2, 2), (3, 5), (64, 128), (67, 131), (1, 300), (300, 1),
             (65, 129), (1080, 1920), (5, 17)]
    kinds = ("shapes", "noise", "blocks", "const")
    hosts = [content(kinds[i % 4], 1, h, w, ch, seed=100 + i)[0] for i, (h, w) in enumerate(sizes)]
    run_list_and_check(hosts, *thr(a), l2, a, rng, ctx=gpu_ctx, name=f"mixed ch={ch}")
    run_list_and_check(hosts[2:], *thr(a), l2, a, rng, ctx=gpu_ctx, name=f"mixed byte staging ch={ch}", aligned=False)


@pytest.mark.parametrize("a", [5, 7])
def test_lists_tall_frame_and_mosaic(gpu_ctx, a):
    """A 1-wide frame taller than the uniform call's grid covers, and outputs that are tiles of one mosaic in rows of their own."""
    import torch
    rng = np.random.default_rng(a)
    for ch in (1, 3):
        tall = content("noise", 1, 70_000, 1, ch, seed=3)[0]
        run_list_and_check([tall, content("shapes", 1, 40, 60, ch, seed=4)[0]], *thr(a), False, a, rng, ctx=gpu_ctx,
                           name=f"tall ch={ch}")
        shapes = [(40, 60), (17, 100), (64, 128), (1, 1), (33, 7)]
        hosts = [content(("shapes", "noise", "blocks")[i % 3], 1, h, w, ch, seed=20 + i)[0] for i, (h, w) in enumerate(shapes)]
        mosaic = torch.full((sum(h for h, _ in shapes) + 3, 160), SENTINEL, dtype=torch.uint8, device="cuda")
        views, y = [], 1
        for i, (h, w) in enumerate(shapes):
            x = 3 * i
            views.append(mosaic[y:y + h, x:x + w])
            y += h
        run_list_and_check(hosts, *thr(a), True, a, rng, ctx=gpu_ctx, name=f"mosaic ch={ch}", outs=views)
        pad = mosaic.cpu().numpy().copy()
        y = 1
        for i, (h, w) in enumerate(shapes):
            pad[y:y + h, 3 * i:3 * i + w] = SENTINEL
            y += h
        assert (pad == SENTINEL).all(), "bytes outside the mosaic tiles were written"


def test_aperture_3_calls_equal_the_existing_calls(gpu_ctx):
    """The new calls with aperture 3 give the existing calls' maps byte for byte, uniform and list."""
    import torch
    lib = _lib.load()
    for ch in (1, 3):
        host = content("shapes", 3, 300, 517, ch, seed=61)
        host[1] = content("noise", 1, 300, 517, ch, seed=62)[0]
        dev = torch.from_numpy(host).cuda()
        n, h, w = host.shape[:3]
        for l2 in (0, 1):
            outs = [torch.full((n, h, w), SENTINEL, dtype=torch.uint8, device="cuda") for _ in range(2)]
            _lib.check(lib.b200_cv_canny_device_strided(gpu_ctx.handle, dev.data_ptr(), ch * w, h * w * ch, n, h, w, ch, C.c_double(20),
                                                      C.c_double(60), l2, outs[0].data_ptr(), w, h * w))
            _lib.check(lib.b200_cv_canny_aperture_device_strided(gpu_ctx.handle, dev.data_ptr(), ch * w, h * w * ch, n, h, w, ch,
                                                               C.c_double(20), C.c_double(60), 3, l2, outs[1].data_ptr(), w, h * w))
            gpu_ctx.synchronize()
            assert torch.equal(outs[0], outs[1])
            assert np.array_equal(outs[0].cpu().numpy()[1], want_map(host[1], 20, 60, bool(l2), 3))
            louts = [[torch.full((h, w), SENTINEL, dtype=torch.uint8, device="cuda") for _ in range(n)] for _ in range(2)]
            descs = [[(dev[i].data_ptr(), ch * w, o[i].data_ptr(), w, h, w) for i in range(n)] for o in louts]
            _lib.check(lib.b200_cv_canny_frames_device(gpu_ctx.handle, frame_list(descs[0]), n, ch, C.c_double(20), C.c_double(60), l2))
            _lib.check(lib.b200_cv_canny_aperture_frames_device(gpu_ctx.handle, frame_list(descs[1]), n, ch, C.c_double(20),
                                                              C.c_double(60), 3, l2))
            gpu_ctx.synchronize()
            for i in range(n):
                assert torch.equal(louts[0][i], louts[1][i])
                assert torch.equal(louts[0][i], outs[0][i])


def test_apertures_and_reference_semantics_alternated(gpu_ctx, oracle):
    """Apertures 3, 5 and 7 and the reference's canny alternated on one context, uniform and list calls."""
    import torch
    rng = np.random.default_rng(41)
    for i in range(6):
        n, h, w = 2, int(rng.integers(2, 300)), int(rng.integers(2, 400))
        host = content(("shapes", "noise", "blocks")[i % 3], n, h, w, 1, seed=50 + i)
        dev = torch.from_numpy(host).cuda()
        l2 = bool(i & 1)
        ref = cb.torch_api.canny(dev, 1.4, 20, 60, ctx=gpu_ctx)
        maps = {a: cb.torch_api.cv_canny(dev, *thr(a), apertureSize=a, L2gradient=l2, ctx=gpu_ctx) for a in (7, 3, 5)}
        lists = {a: cb.torch_api.cv_canny_list([dev[0], dev[1, 1:, 1:]], *thr(a), apertureSize=a, L2gradient=l2, ctx=gpu_ctx)
                 for a in (5, 7, 3)}
        ref2 = cb.torch_api.canny(dev, 1.0, 0, 30, ctx=gpu_ctx)
        torch.cuda.synchronize()
        for f in range(n):
            assert np.array_equal(ref.cpu().numpy()[f].astype(np.int16), oracle.canny(host[f], 1.4, 20, 60)), (i, f)
            assert np.array_equal(ref2.cpu().numpy()[f].astype(np.int16), oracle.canny(host[f], 1.0, 0, 30)), (i, f)
            for a in (3, 5, 7):
                assert np.array_equal(maps[a].cpu().numpy()[f], want_map(host[f], *thr(a), l2, a)), (i, f, a)
        for a in (3, 5, 7):
            assert np.array_equal(lists[a][0].cpu().numpy(), want_map(host[0], *thr(a), l2, a)), (i, a)
            assert np.array_equal(lists[a][1].cpu().numpy(), want_map(np.ascontiguousarray(host[1, 1:, 1:]), *thr(a), l2, a)), (i, a)


def test_non_default_stream(gpu_ctx):
    import torch
    host = content("shapes", 3, 260, 400, 3, seed=31)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        dev = torch.from_numpy(host).cuda(non_blocking=False)
        res = {a: cb.torch_api.cv_canny_color(dev, *thr(a), apertureSize=a, L2gradient=a == 7, ctx=gpu_ctx) for a in (5, 7)}
        lst = cb.torch_api.cv_canny_color_list([dev[0], dev[2]], *thr(7), apertureSize=7, ctx=gpu_ctx)
    s.synchronize()
    for f in range(3):
        for a in (5, 7):
            assert np.array_equal(res[a].cpu().numpy()[f], want_map(host[f], *thr(a), a == 7, a))
    assert np.array_equal(lst[1].cpu().numpy(), want_map(host[2], *thr(7), False, 7))


def test_aperture_7_thresholds_and_bad_apertures(gpu_ctx):
    import torch
    host = content("noise", 2, 64, 64, 1, seed=64)
    dev = torch.from_numpy(host).cuda()
    # 600000 / 16 is clamped to 32767, whose square is above every magnitude; 2^34 / 16 fits in int32
    for lo, hi, l2 in ((10, 600000, True), (2.0 ** 34, 2.0 ** 34, False), (0, 0, False), (-5, 2.0 ** 34, True), (16 * 2047, 16 * 2048, True)):
        res = run_and_check(dev, host, lo, hi, l2, 7, ctx=gpu_ctx, name="aperture 7 thresholds")
        if hi >= 600000:
            assert not res.any()
    with pytest.raises(cb.CannyB200Error):   # 2^35 / 16 = 2^31 does not fit in int32
        cb.torch_api.cv_canny(dev, 10, 2.0 ** 35, apertureSize=7, ctx=gpu_ctx)
    for a in (1, 2, 4, 6, 8, 9, 0, -1):
        with pytest.raises(cb.CannyB200Error, match="aperture"):
            cb.torch_api.cv_canny(dev, 20, 60, apertureSize=a, ctx=gpu_ctx)
        with pytest.raises(cb.CannyB200Error, match="aperture"):
            cb.torch_api.cv_canny_list([dev[0]], 20, 60, apertureSize=a, ctx=gpu_ctx)
    run_and_check(dev, host, 20, 60, False, 3, ctx=gpu_ctx, name="after the rejections")


def test_seeded_fuzz(gpu_ctx):
    """120 seeded cases across apertures 3, 5 and 7: sizes, channel counts, L1 / L2, layouts (dense, aligned crop, unaligned crop),
    contents and thresholds around each aperture's magnitudes."""
    import torch
    rng = np.random.default_rng(20261022)
    for i in range(120):
        a = (3, 5, 7)[i % 3]
        ch = int(rng.choice([1, 3]))
        n = int(rng.integers(1, 4))
        h, w = int(rng.integers(1, 200)), int(rng.integers(1, 300))
        l2 = bool(rng.integers(0, 2))
        kind = ("shapes", "noise", "const", "blocks")[int(rng.integers(0, 4))]
        host = content(kind, n, h, w, ch, seed=1000 + i)
        lo, hi = float(rng.uniform(-20, 300)) * SCALE[a], float(rng.uniform(-20, 600)) * SCALE[a]
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
        run_and_check(dev, host, lo, hi, l2, a, out=buf[:, :h, :w], ctx=gpu_ctx, name=f"fuzz {i} a={a} {kind} {n}x{h}x{w}x{ch}")
        check_padding(buf, n, h, w, f"fuzz {i}")
