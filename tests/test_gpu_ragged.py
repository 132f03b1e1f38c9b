"""Ragged frame lists on the B200 (b200_canny_frames_device, torch_api.canny_list): frames of different sizes and layouts in one
call, every map against the oracle bit for bit, output padding filled with a sentinel that must survive."""
import numpy as np
import pytest

import canny_edge_b200 as cb
from canny_edge_b200 import torch_api

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5


def gray_formula(bgr):
    b, g, r = (bgr[..., i].astype(np.int64) for i in range(3))
    return ((b * 3735 + g * 19235 + r * 9798 + (1 << 14)) >> 15).astype(np.uint8)


def synth(h, w, seed, kind=0):
    return cb.synth_host(1, h, w, kind=kind, seed=seed)[0]


class Frame:
    """A host frame and its device view: `x0` leading bytes per row and `pad` trailing ones (random), so the view's base and pitch
    are 16-byte aligned (TMA staging) or not (byte staging) as the case wants; its output is a view into a sentinel-filled buffer."""

    def __init__(self, host, rng, x0=0, pad=0, out_x0=0, out_pad=0, bgr=None):
        import torch
        self.host = host                     # gray frame the oracle sees
        h, w = host.shape
        src = host if bgr is None else bgr.reshape(h, 3 * w)
        bpp = 1 if bgr is None else 3
        buf = rng.integers(0, 256, (h + 1, x0 + bpp * w + pad), dtype=np.uint8)
        buf[:h, x0:x0 + bpp * w] = src
        d = torch.from_numpy(buf).cuda()
        self.view = d[:h, x0:x0 + bpp * w] if bgr is None else d[:h, x0:x0 + 3 * w].view(h, w, 3)
        self.out_buf = torch.full((h + 1, out_x0 + w + out_pad), SENTINEL, dtype=torch.uint8, device="cuda")
        self.out = self.out_buf[:h, out_x0:out_x0 + w]
        self.out_x0 = out_x0


def check(oracle, frames, sigma, lo, hi, name, outs=None):
    for i, f in enumerate(frames):
        h, w = f.host.shape
        want = oracle.canny(f.host, sigma, lo, hi)
        got = (outs[i] if outs is not None else f.out).cpu().numpy()
        diff = int((got.astype(np.int16) != want).sum())
        assert diff == 0, f"{name}: frame {i} ({h}x{w}) differs in {diff} pixels"
        if outs is None:
            pad = f.out_buf.cpu().numpy()
            pad[:h, f.out_x0:f.out_x0 + w] = SENTINEL
            assert (pad == SENTINEL).all(), f"{name}: frame {i}: bytes outside the map were written"


def run(frames, sigma, lo, hi, ctx=None, bgr=False):
    import torch
    fn = torch_api.canny_bgr_list if bgr else torch_api.canny_list
    res = fn([f.view for f in frames], sigma, lo, hi, out=[f.out for f in frames], ctx=ctx)
    torch.cuda.synchronize()
    assert all(r is f.out for r, f in zip(res, frames))


def mixed_frames(rng, seed):
    sizes = [(2, 2), (2, 37), (41, 2), (3, 3), (256, 256), (480, 640)] + [(int(rng.integers(2, 120)), w) for w in range(3, 302, 14)]
    sizes += [(int(rng.integers(20, 200)), 16 * k) for k in (1, 4, 9, 40)]
    frames = []
    for i, (h, w) in enumerate(sizes):
        tma = i % 2 == 0
        frames.append(Frame(synth(h, w, seed + i, kind=i % 2), rng, x0=0 if tma else int(rng.choice([1, 3, 7])),
                            pad=(-w) % 16 + 16 * int(rng.integers(0, 2)) if tma else int(rng.integers(0, 5)),
                            out_x0=int(rng.integers(0, 5)), out_pad=int(rng.integers(0, 5))))
    return frames


def test_mixed_sizes_and_staging_forms(gpu_ctx, oracle):
    rng = np.random.default_rng(1)
    frames = mixed_frames(rng, 100)
    run(frames, 1.4, 20, 60, ctx=gpu_ctx)
    check(oracle, frames, 1.4, 20, 60, "mixed")


def test_4k_next_to_small(gpu_ctx, oracle):
    rng = np.random.default_rng(2)
    frames = [Frame(synth(256, 256, 5), rng), Frame(synth(2160, 3840, 6), rng), Frame(synth(256, 256, 7, 1), rng, x0=3),
              Frame(synth(2160, 3840, 8, 1), rng, x0=5, out_x0=1)]
    run(frames, 1.4, 20, 60, ctx=gpu_ctx)
    check(oracle, frames, 1.4, 20, 60, "4k")


@pytest.mark.parametrize("sigma", [0.5, 0.8, 1.4, 2.0, 3.0, 5.0, 2.4, 0.1])
def test_sigmas(oracle, sigma):
    """Half-windows 2, 3, 5, 6, 9, 15 (ragged kernels), 8 (sigma 2.4: no front3 build) and a sigma whose weights are `tiny`: the
    last two take the strided path frame by frame, which the front-kernel counters show."""
    ctx = cb.Context(0)
    try:
        rng = np.random.default_rng(int(sigma * 10))
        frames = [Frame(synth(h, w, int(sigma * 100) + i, i % 2), rng, x0=(i % 2) * 3)
                  for i, (h, w) in enumerate([(200, 333), (70, 64), (131, 517), (2, 9)])]
        run(frames, sigma, 20, 60, ctx=ctx)
        check(oracle, frames, sigma, 20, 60, f"sigma={sigma}")
        fast, gen = ctx.front_kernel_stats()
        if sigma in (2.4, 0.1):
            assert gen == 4 and fast == 0, (fast, gen)
        else:
            assert gen == 0 and 1 <= fast <= 2, (fast, gen)   # one launch per staging form
    finally:
        ctx.close()


@pytest.mark.parametrize("lo,hi", [(0, 60), (-5, 40), (-10, -1), (20, 300), (60, 20), (40, 40), (0, 0)])
def test_thresholds(gpu_ctx, oracle, lo, hi):
    rng = np.random.default_rng(1000 + lo * 7 + hi)
    frames = [Frame(synth(h, w, 300 + i, i % 2), rng, x0=i % 2) for i, (h, w) in enumerate([(90, 170), (33, 47), (128, 256)])]
    run(frames, 1.4, lo, hi, ctx=gpu_ctx)
    check(oracle, frames, 1.4, lo, hi, f"thresholds {lo}/{hi}")


def test_unsupported_thresholds(gpu_ctx):
    rng = np.random.default_rng(3)
    f = Frame(synth(20, 20, 1), rng)
    with pytest.raises(cb.CannyB200Error, match="status 4"):
        torch_api.canny_list([f.view], 1.4, 300, 100, ctx=gpu_ctx)


def test_noise_frames_dense_list(gpu_ctx, oracle):
    """Uniform noise: a large share of the pixels are weak, and the list-driven kernels take them all."""
    rng = np.random.default_rng(4)
    frames = []
    for i, (h, w) in enumerate([(300, 400), (97, 501), (256, 256), (5, 640)]):
        frames.append(Frame(rng.integers(0, 256, (h, w), dtype=np.uint8), rng, x0=(i % 2) * 5))
    for lo, hi in ((20, 60), (5, 250), (0, 200)):
        run(frames, 1.4, lo, hi, ctx=gpu_ctx)
        check(oracle, frames, 1.4, lo, hi, f"noise {lo}/{hi}")


def test_quirk_in_later_frames(gpu_ctx, oracle):
    """The reference's one-way link (0,1) -> (1,0) in frames that are not first in the list: (0,1) strong and (1,0) weak, and the
    other way round."""
    rng = np.random.default_rng(5)
    frames = []
    for i in range(6):
        img = np.zeros((40, 50), np.uint8)
        if i % 2 == 0:
            img[0, 1:] = 255          # a strong edge along the top row, reaching (0,1)
            img[3:, 0] = 60           # a weak run down column 0
        else:
            img[1:, 0] = 255
            img[0, 3:] = 60
        frames.append(Frame(img, rng, x0=(i % 3) * 16 + (i % 2)))
    frames.insert(0, Frame(synth(64, 80, 9), rng))
    for lo, hi in ((20, 60), (1, 200), (10, 100)):
        run(frames, 0.5, lo, hi, ctx=gpu_ctx)
        check(oracle, frames, 0.5, lo, hi, f"quirk {lo}/{hi}")


def test_chunks_by_frame_cap_and_by_pixels(oracle):
    ctx = cb.Context(0)
    try:
        rng = np.random.default_rng(6)
        frames = mixed_frames(rng, 500)[:14]
        ctx.set_chunk_frames(3)          # 5 chunks over three slots
        run(frames, 1.4, 20, 60, ctx=ctx)
        check(oracle, frames, 1.4, 20, 60, "chunk_frames=3")
        ctx.set_chunk_frames(0)
        # by pixel volume: 4K frames (8.3 Mpix) fill a 75 Mpix chunk at 9; a 12000 x 8000 frame (96 Mpix) is above the budget and
        # has a chunk of its own
        big = [Frame(synth(2160, 3840, 600 + i, i % 2), rng, x0=(i % 4 == 3) * 3) for i in range(11)]
        huge = Frame(synth(8000, 12000, 700), rng)
        small = [Frame(synth(100, 130, 800 + i), rng) for i in range(3)]
        frames = big[:5] + [huge] + small + big[5:]
        run(frames, 1.4, 20, 60, ctx=ctx)
        check(oracle, frames, 1.4, 20, 60, "chunks by pixels")
    finally:
        ctx.close()


def test_mosaic_output(gpu_ctx, oracle):
    """Outputs as tiles of one mosaic tensor, each tile in rows of its own at its own column; everything else must survive."""
    import torch
    rng = np.random.default_rng(7)
    sizes = [(60, 100), (33, 250), (80, 17), (2, 300), (45, 45)]
    hosts = [synth(h, w, 900 + i, i % 2) for i, (h, w) in enumerate(sizes)]
    mosaic = torch.full((sum(h for h, _ in sizes) + 3, 320), SENTINEL, dtype=torch.uint8, device="cuda")
    outs, y, cols = [], 1, []
    for (h, w) in sizes:
        x = int(rng.integers(0, 320 - w + 1))
        outs.append(mosaic[y:y + h, x:x + w])
        cols.append((y, x))
        y += h
    ins = [torch.from_numpy(hh).cuda() for hh in hosts]
    torch_api.canny_list(ins, 1.4, 20, 60, out=outs, ctx=gpu_ctx)
    torch.cuda.synchronize()
    got = mosaic.cpu().numpy()
    rest = got.copy()
    for hh, (y, x) in zip(hosts, cols):
        h, w = hh.shape
        assert (got[y:y + h, x:x + w].astype(np.int16) == oracle.canny(hh, 1.4, 20, 60)).all(), (h, w)
        rest[y:y + h, x:x + w] = SENTINEL
    assert (rest == SENTINEL).all()


def test_same_shape_list_equals_strided_batch(gpu_ctx):
    import torch
    n, h, w = 6, 540, 961
    host = np.stack([synth(h, w, 1000 + i, i % 2) for i in range(n)])
    buf = torch.from_numpy(np.pad(host, ((0, 0), (0, 0), (3, 20)))).cuda()
    d_in = buf[:, :, 3:3 + w]
    a = torch.zeros((n, h, w + 7), dtype=torch.uint8, device="cuda")
    b = torch.zeros_like(a)
    torch.cuda.synchronize()
    cb.canny_batch_device_strided_ptr(gpu_ctx, d_in.data_ptr(), d_in.stride(1), d_in.stride(0), n, h, w, 1.4, 20, 60,
                                      a.data_ptr(), a.stride(1), a.stride(0))
    gpu_ctx.synchronize()
    descs = [(d_in[i].data_ptr(), d_in.stride(1), b[i].data_ptr(), b.stride(1), h, w) for i in range(n)]
    cb.canny_frames_device_ptr(gpu_ctx, descs, 1.4, 20, 60)
    gpu_ctx.synchronize()
    assert torch.equal(a, b)
    dense = torch.from_numpy(host).cuda()
    c, d = torch.empty_like(dense), torch.empty_like(dense)
    torch.cuda.synchronize()
    cb.canny_batch_device_ptr(gpu_ctx, dense.data_ptr(), n, h, w, 1.4, 20, 60, c.data_ptr())
    gpu_ctx.synchronize()
    cb.canny_frames_device_ptr(gpu_ctx, [(dense[i].data_ptr(), w, d[i].data_ptr(), w, h, w) for i in range(n)], 1.4, 20, 60)
    gpu_ctx.synchronize()
    assert torch.equal(c, d)


@pytest.mark.parametrize("sigma", [1.4, 5.0, 2.4])
def test_bgr_lists(gpu_ctx, oracle, sigma):
    rng = np.random.default_rng(int(sigma * 10) + 11)
    frames = []
    for i, (h, w) in enumerate([(100, 160), (77, 123), (2, 2), (64, 640), (31, 33)]):
        bgr = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        bgr[..., 1] = synth(h, w, 1100 + i, i % 2)
        frames.append(Frame(gray_formula(bgr), rng, x0=(i % 2) * 5, pad=int(rng.integers(0, 9)), bgr=bgr, out_x0=i % 3))
    run(frames, sigma, 20, 60, ctx=gpu_ctx, bgr=True)
    check(oracle, frames, sigma, 20, 60, f"bgr sigma={sigma}")


def test_non_default_stream_and_two_streams(oracle):
    import torch
    rng = np.random.default_rng(12)
    lists = [[synth(int(rng.integers(2, 400)), int(rng.integers(2, 700)), 1200 + 10 * k + i, (k + i) % 2) for i in range(5)]
             for k in range(6)]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(s1):
        d = [torch.from_numpy(hh).cuda() for hh in lists[0]]
        res = [r.clone() for r in torch_api.canny_list(d, 1.4, 20, 60)]
    s1.synchronize()
    for hh, r in zip(lists[0], res):
        assert (r.cpu().numpy().astype(np.int16) == oracle.canny(hh, 1.4, 20, 60)).all()
    d_in = [[torch.from_numpy(hh).cuda() for hh in lst] for lst in lists]
    torch.cuda.synchronize()
    outs = []
    for k, d in enumerate(d_in):
        st = s1 if k % 2 == 0 else s2
        st.wait_stream(torch.cuda.default_stream())
        with torch.cuda.stream(st):
            outs.append(torch_api.canny_list(d, 1.4, 20, 60))
    torch.cuda.synchronize()
    for lst, o in zip(lists, outs):
        for hh, r in zip(lst, o):
            assert (r.cpu().numpy().astype(np.int16) == oracle.canny(hh, 1.4, 20, 60)).all()


def test_mixed_devices_rejected():
    import torch
    a = torch.zeros((20, 30), dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError, match="CUDA"):
        torch_api.canny_list([a, a.cpu()], 1.4, 20, 60)
    with pytest.raises(ValueError, match="CUDA"):
        torch_api.canny_list([a], 1.4, 20, 60, out=[torch.zeros((20, 30), dtype=torch.uint8)])


def test_fuzz_lists(oracle):
    import torch
    rng = np.random.default_rng(2025)
    ctx = cb.Context(0)
    try:
        for case in range(100):
            n = int(rng.integers(1, 41))
            sigma = float(rng.choice([0.5, 0.8, 1.0, 1.4, 2.0, 3.0, 5.0]))
            lo = int(rng.integers(-5, 80))
            hi = int(lo + rng.integers(-10, 100))
            frames = []
            for i in range(n):
                h, w = int(rng.integers(2, 150)), int(rng.integers(2, 330))
                tma = rng.random() < 0.5
                frames.append(Frame(synth(h, w, case * 100 + i, int(rng.integers(0, 2))), rng,
                                    x0=int(rng.choice([0, 16])) if tma else int(rng.integers(1, 16)),
                                    pad=(-w) % 16 if tma else int(rng.integers(0, 20)),
                                    out_x0=int(rng.integers(0, 4)), out_pad=int(rng.integers(0, 4))))
            ctx.set_chunk_frames(int(rng.choice([0, 0, 1, 7])))
            run(frames, sigma, lo, hi, ctx=ctx)
            check(oracle, frames, sigma, lo, hi, f"case {case} n={n} sigma={sigma} {lo}/{hi}")
    finally:
        ctx.close()
