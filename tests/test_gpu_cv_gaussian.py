"""cv::Canny of a Gaussian-blurred frame on the B200 (torch_api.cv_canny / cv_canny_color / cv_canny_list / cv_canny_color_list with
gaussian=, b200_cv_gaussian_canny_device_strided and b200_cv_gaussian_canny_frames_device): every map against the numpy restatement
(tests/cv_gaussian_ref.py + tests/cv_canny_aperture_ref.py) bit for bit, and against cv2.Canny(cv2.GaussianBlur(...)) where cv2 is
importable.  Every radius class (none, <= 3, <= 15), asymmetric kernels, frames smaller than the kernel, tile edges, 16-byte and
byte staging; outputs sit in sentinel-filled buffers whose padding must survive."""
import numpy as np
import pytest

import canny_edge_b200 as cb
from cv_canny_aperture_ref import cv_canny
from cv_gaussian_ref import cv2_gaussian_blur, gaussian_blur
from test_gpu_cv_canny import check_padding, content, sentinel_like
from test_gpu_cv_ragged import Outs, place

pytestmark = pytest.mark.gpu

try:
    import cv2
except Exception:   # cv2 is optional: the restatement is the specification
    cv2 = None

SCALE = {3: 1, 5: 16, 7: 256}
# (ksize, sigmaX, sigmaY): radius class <= 3, then <= 15, asymmetric ones, a derived size, the largest
BLURS = [((3, 3), 0.0, 0.0), ((5, 5), 0.0, 0.0), ((7, 7), 1.2, 0.0), ((1, 5), 0.0, 0.0), ((0, 0), 1.4, 0.0), ((0, 0), 2.0, 0.0),
         ((31, 31), 0.0, 0.0), ((31, 3), 0.0, 0.0), ((5, 25), 2.5, 0.7), ((9, 1), 0.0, 0.0)]


def want_map(img, blur, lo, hi, l2, a):
    ksize, sx, sy = blur
    want = cv_canny(gaussian_blur(img, ksize, sx, sy), lo, hi, l2, a)
    if cv2 is not None:
        got = cv2.Canny(cv2_gaussian_blur(cv2, img, ksize, sx, sy), lo, hi, apertureSize=a, L2gradient=l2)
        assert np.array_equal(want, got), "restatement != cv2"
    return want


def run_and_check(frames_dev, host, blur, lo, hi, l2, a, out=None, ctx=None, name=""):
    """frames_dev: CUDA view of `host` ((N, H, W) or (N, H, W, 3)); out: a view into a sentinel buffer, or None."""
    import torch
    fn = cb.torch_api.cv_canny_color if host.ndim == 4 else cb.torch_api.cv_canny
    res = fn(frames_dev, lo, hi, apertureSize=a, L2gradient=l2, gaussian=blur, out=out, ctx=ctx)
    torch.cuda.synchronize()
    got = res.cpu().numpy()
    for f in range(host.shape[0]):
        diff = int((got[f] != want_map(host[f], blur, lo, hi, l2, a)).sum())
        assert diff == 0, f"{name}: frame {f} (blur {blur}, aperture {a}, l2={l2}, {lo}, {hi}) differs in {diff} pixels"
    return res


def run_list_and_check(hosts, blur, lo, hi, l2, a, rng, ctx=None, name="", aligned=None):
    import torch
    devs = [place(x, (i % 2 == 0) if aligned is None else aligned, rng) for i, x in enumerate(hosts)]
    outs = Outs([x.shape[:2] for x in hosts], rng)
    fn = cb.torch_api.cv_canny_color_list if hosts[0].ndim == 3 else cb.torch_api.cv_canny_list
    res = fn(devs, lo, hi, apertureSize=a, L2gradient=l2, gaussian=blur, out=outs.views, ctx=ctx)
    torch.cuda.synchronize()
    assert all(r is v for r, v in zip(res, outs.views))
    for i, (x, r) in enumerate(zip(hosts, res)):
        diff = int((r.cpu().numpy() != want_map(x, blur, lo, hi, l2, a)).sum())
        assert diff == 0, f"{name}: frame {i} {x.shape} (blur {blur}, aperture {a}, l2={l2}) differs in {diff} pixels"
    outs.check_padding(name)
    return res


def _noisy(kind, n, h, w, ch, seed):
    host = content(kind, n, h, w, ch, seed=seed)
    if kind == "shapes":   # a noise band, so that blurred frames keep weak and strong pixels
        band = host[:, h // 3:h // 2]
        host[:, h // 3:h // 2] = np.random.default_rng(seed).integers(0, 256, band.shape, dtype=np.uint8)
    return host


@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("bi", range(len(BLURS)))
def test_small_sizes_and_tile_edges(gpu_ctx, bi, ch):
    """Frames from 1 x 1, narrower and shorter than the kernel, and around the 128 x 64 tile edges plus the radius."""
    import torch
    blur = BLURS[bi]
    sizes = [(1, 1), (1, 37), (45, 1), (2, 2), (3, 5), (7, 13), (13, 7), (63, 127), (64, 128), (65, 129), (79, 143), (49, 113),
             (130, 255)]
    for i, (h, w) in enumerate(sizes):
        a = (3, 5, 7)[(i + bi) % 3]
        l2 = (i + bi + ch) % 2 == 1
        kind = ("noise", "shapes", "blocks")[i % 3]
        host = _noisy(kind, 2, h, w, ch, seed=h * 1000 + w + bi)
        buf = sentinel_like(2, h, w, w + 5, 1)
        lo, hi = 10 * SCALE[a], 30 * SCALE[a]
        run_and_check(torch.from_numpy(host).cuda(), host, blur, lo, hi, l2, a, out=buf[:, :h, :w], ctx=gpu_ctx,
                      name=f"{kind} {h}x{w}x{ch}")
        check_padding(buf, 2, h, w, f"{kind} {h}x{w}x{ch}")


@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("blur", [((5, 5), 0.0, 0.0), ((0, 0), 2.0, 0.0), ((31, 31), 0.0, 0.0), ((3, 21), 0.0, 0.0)])
def test_lists(gpu_ctx, blur, ch):
    """Frames of different sizes in one call, 16-byte and byte staging in one list."""
    rng = np.random.default_rng(31 + ch)
    sizes = [(1, 1), (5, 3), (14, 31), (64, 128), (65, 129), (63, 127), (200, 333), (1, 300), (300, 1), (97, 160)]
    hosts = [_noisy(("noise", "shapes", "blocks")[i % 3], 1, h, w, ch, seed=i)[0] for i, (h, w) in enumerate(sizes)]
    for l2, a in ((False, 3), (True, 5), (False, 7)):
        run_list_and_check(hosts, blur, 10 * SCALE[a], 30 * SCALE[a], l2, a, rng, ctx=gpu_ctx, name=f"list {blur} a{a}")


@pytest.mark.parametrize("blur", [((5, 5), 0.0, 0.0), ((0, 0), 1.4, 0.0), ((31, 31), 0.0, 0.0)])
def test_crops_pitches_and_channel_views(gpu_ctx, blur):
    """Strided crops, unaligned bases and pitches (byte staging) next to aligned ones (16-byte staging)."""
    import torch
    rng = np.random.default_rng(2)
    big = content("shapes", 2, 400, 700, 1, seed=8)
    big[:, 100:180] = rng.integers(0, 256, big[:, 100:180].shape, dtype=np.uint8)
    dev = torch.from_numpy(big).cuda()
    for (y0, y1, x0, x1) in ((16, 300, 32, 672), (3, 397, 5, 690), (1, 2, 7, 600), (10, 300, 699, 700)):
        host = np.ascontiguousarray(big[:, y0:y1, x0:x1])
        h, w = host.shape[1:]
        buf = sentinel_like(2, h, w, w + 7, 3)
        run_and_check(dev[:, y0:y1, x0:x1], host, blur, 20, 60, False, 3, out=buf[:, :h, :w], ctx=gpu_ctx,
                      name=f"crop {(y0, y1, x0, x1)}")
        check_padding(buf, 2, h, w, "crop")
    for pitch in (720, 701):
        padded = torch.zeros((2, 400, pitch), dtype=torch.uint8, device="cuda")
        padded[:, :, :700] = dev
        run_and_check(padded[:, :, :700], big, blur, 20, 60, True, 5 if pitch == 720 else 3, ctx=gpu_ctx, name=f"pitch {pitch}")
    col = content("shapes", 2, 300, 500, 3, seed=9)
    col[:, 50:90] = rng.integers(0, 256, col[:, 50:90].shape, dtype=np.uint8)
    dcol = torch.from_numpy(col).cuda()
    for (y0, y1, x0, x1) in ((0, 300, 16, 496), (7, 250, 3, 499), (1, 300, 0, 1)):
        host = np.ascontiguousarray(col[:, y0:y1, x0:x1])
        h, w = host.shape[1:3]
        buf = sentinel_like(2, h, w, w + 9, 1)
        run_and_check(dcol[:, y0:y1, x0:x1], host, blur, 20, 60, True, 3, out=buf[:, :h, :w], ctx=gpu_ctx,
                      name=f"color crop {(y0, y1, x0, x1)}")
        check_padding(buf, 2, h, w, "color crop")


@pytest.mark.parametrize("ch", [1, 3])
def test_4k_frame(gpu_ctx, ch):
    import torch
    host = _noisy("shapes", 1, 2160, 3840, ch, seed=5)
    dev = torch.from_numpy(host).cuda()
    for blur, a, l2 in ((((5, 5), 0.0, 0.0), 3, False), (((0, 0), 2.0, 0.0), 5, True), (((31, 31), 0.0, 0.0), 3, False)):
        run_and_check(dev, host, blur, 20 * SCALE[a], 60 * SCALE[a], l2, a, ctx=gpu_ctx, name=f"4K x{ch} {blur}")


def test_multi_chunk():
    """More frames than one chunk: the blur parameters reach every chunk's launch on every stream slot."""
    import torch
    c = cb.Context(0)
    try:
        c.set_chunk_frames(2)
        host = _noisy("shapes", 7, 150, 260, 3, seed=3)
        run_and_check(torch.from_numpy(host).cuda(), host, ((0, 0), 1.4, 0.0), 20, 60, False, 3, ctx=c, name="chunks")
        hosts = [x for x in host] + [host[0, :77, :91]]
        run_list_and_check(hosts, ((9, 5), 0.0, 0.0), 20, 60, True, 3, np.random.default_rng(4), ctx=c, name="list chunks")
    finally:
        c.close()


@pytest.mark.parametrize("ch", [1, 3])
def test_identity_and_no_blur(gpu_ctx, ch):
    """ksize (1, 1) gives cv_canny's maps (the unblurred kernels run); gaussian=None is the call without the keyword."""
    import torch
    host = _noisy("shapes", 2, 130, 300, ch, seed=11)
    dev = torch.from_numpy(host).cuda()
    fn = cb.torch_api.cv_canny_color if ch == 3 else cb.torch_api.cv_canny
    lfn = cb.torch_api.cv_canny_color_list if ch == 3 else cb.torch_api.cv_canny_list
    for a in (3, 5, 7):
        lo, hi = 20 * SCALE[a], 60 * SCALE[a]
        plain = fn(dev, lo, hi, apertureSize=a, ctx=gpu_ctx).cpu()
        for g in (((1, 1), 0.0), ((1, 1), 3.0, 2.0), None):
            assert torch.equal(fn(dev, lo, hi, apertureSize=a, gaussian=g, ctx=gpu_ctx).cpu(), plain), (a, g)
            got = lfn([dev[0], dev[1, 5:, 7:]], lo, hi, apertureSize=a, gaussian=g, ctx=gpu_ctx)
            assert torch.equal(got[0].cpu(), plain[0]), (a, g)
            want = lfn([dev[1, 5:, 7:]], lo, hi, apertureSize=a, ctx=gpu_ctx)[0]
            assert torch.equal(got[1].cpu(), want.cpu()), (a, g)
        blurred = fn(dev, lo, hi, apertureSize=a, gaussian=((5, 5), 0), ctx=gpu_ctx).cpu()
        assert not torch.equal(blurred, plain)


def test_rejections_on_the_device_path(gpu_ctx):
    """Values cv2 rejects come back from the library before any device work, on a real device too."""
    import torch
    x = torch.zeros((2, 32, 48), dtype=torch.uint8, device="cuda")
    for g, status in ((((4, 4), 0), cb._lib.ERR_INVALID_ARG), (((0, 0), 0), cb._lib.ERR_INVALID_ARG),
                      (((5, 5), float("nan")), cb._lib.ERR_INVALID_ARG), (((33, 33), 0), cb._lib.ERR_UNSUPPORTED)):
        with pytest.raises(cb.CannyB200Error) as e:
            cb.torch_api.cv_canny(x, 20, 60, gaussian=g, ctx=gpu_ctx)
        assert e.value.status == status
        with pytest.raises(cb.CannyB200Error) as e:
            cb.torch_api.cv_canny_list([x[0], x[1]], 20, 60, gaussian=g, ctx=gpu_ctx)
        assert e.value.status == status
