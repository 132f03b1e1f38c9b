"""Strided device batches on the B200: pitched and cropped inputs, pitched outputs whose padding must survive byte for byte, every
frame against the oracle."""
import numpy as np
import pytest

import canny_edge_b200 as cb
from canny_edge_b200._lib import load

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5


def gray_formula(bgr):
    b, g, r = (bgr[..., i].astype(np.int64) for i in range(3))
    return ((b * 3735 + g * 19235 + r * 9798 + (1 << 14)) >> 15).astype(np.uint8)


def frames_of(n, h, w, seed, kinds=(0, 1)):
    out = np.empty((n, h, w), np.uint8)
    for f in range(n):
        out[f] = cb.synth_host(1, h, w, kind=kinds[f % len(kinds)], seed=seed + f)[0]
    return out


def padded_input(host, pitch, fpad, rng):
    """Device tensor (n, h, pitch) plus fpad rows of random bytes per frame; the frames sit in columns [0, w)."""
    import torch
    n, h, w = host.shape
    buf = rng.integers(0, 256, (n, h + fpad, pitch), dtype=np.uint8)
    buf[:, :h, :w] = host
    return torch.from_numpy(buf).cuda()


def sentinel_output(n, h, pitch, fpad):
    import torch
    return torch.full((n, h + fpad, pitch), SENTINEL, dtype=torch.uint8, device="cuda")


def check_result(oracle, host_gray, out_buf, h, w, sigma, lo, hi, name):
    got = out_buf.cpu().numpy()
    for f in range(host_gray.shape[0]):
        want = oracle.canny(host_gray[f], sigma, lo, hi)
        diff = int((got[f, :h, :w].astype(np.int16) != want).sum())
        assert diff == 0, f"{name}: frame {f} differs in {diff} pixels"
    pad = got.copy()
    pad[:, :h, :w] = SENTINEL
    assert (pad == SENTINEL).all(), f"{name}: bytes outside the frames were written"


def run_gray(ctx, d_in, d_out, n, h, w, sigma, lo, hi):
    import torch
    torch.cuda.synchronize()
    cb.canny_batch_device_strided_ptr(ctx, d_in.data_ptr(), d_in.stride(1), d_in.stride(0), n, h, w, sigma, lo, hi,
                                      d_out.data_ptr(), d_out.stride(1), d_out.stride(0))
    ctx.synchronize()


@pytest.mark.parametrize("w", [641, 648, 652, 3840])
@pytest.mark.parametrize("pad", ["tma", "odd"])
def test_padded_pitches(gpu_ctx, oracle, w, pad):
    rng = np.random.default_rng(w)
    n, h = 3, 270 if w < 1000 else 300
    host = frames_of(n, h, w, seed=w)
    in_pitch = ((w + 15) // 16 + 1) * 16 if pad == "tma" else w + 7    # a multiple of 16 (TMA staging) or an odd one
    out_pitch = w + (12 if pad == "tma" else 5)
    d_in = padded_input(host, in_pitch, 2, rng)
    d_out = sentinel_output(n, h, out_pitch, 3)
    run_gray(gpu_ctx, d_in, d_out, n, h, w, 1.4, 20, 60)
    check_result(oracle, host, d_out, h, w, 1.4, 20, 60, f"w={w} pad={pad}")


@pytest.mark.parametrize("sigma", [0.5, 0.8, 1.4, 2.0, 3.0, 5.0, 2.4])
def test_sigmas(gpu_ctx, oracle, sigma):
    # half-windows 2, 3, 5, 6, 9 (front3), 15 (sigma 5) and 8 (sigma 2.4: the generic kernel)
    rng = np.random.default_rng(int(sigma * 10))
    n, h, w = 2, 200, 333
    host = frames_of(n, h, w, seed=int(sigma * 100))
    for in_pitch, out_pitch in ((352, 340), (341, 333)):
        d_in = padded_input(host, in_pitch, 1, rng)
        d_out = sentinel_output(n, h, out_pitch, 2)
        run_gray(gpu_ctx, d_in, d_out, n, h, w, sigma, 20, 60)
        check_result(oracle, host, d_out, h, w, sigma, 20, 60, f"sigma={sigma} pitch={in_pitch}/{out_pitch}")


def test_torch_crops_and_channels(oracle):
    import torch
    from canny_edge_b200 import torch_api
    big = frames_of(4, 300, 700, seed=3)
    d_big = torch.from_numpy(big).cuda()
    for y0, x0 in ((16, 32), (5, 13)):                 # aligned and unaligned column offsets
        crop = d_big[:, y0:y0 + 250, x0:x0 + 600]
        out_big = torch.full((4, 300, 700), SENTINEL, dtype=torch.uint8, device="cuda")
        out_view = out_big[:, 20:270, 50:650]
        torch_api.canny(crop, 1.4, 20, 60, out=out_view)
        torch.cuda.synchronize()
        got = out_big.cpu().numpy()
        for f in range(4):
            want = oracle.canny(np.ascontiguousarray(big[f, y0:y0 + 250, x0:x0 + 600]), 1.4, 20, 60)
            assert (got[f, 20:270, 50:650].astype(np.int16) == want).all(), (y0, x0, f)
        rest = got.copy()
        rest[:, 20:270, 50:650] = SENTINEL
        assert (rest == SENTINEL).all()
        single = torch_api.canny(crop[2], 1.4, 20, 60)
        torch.cuda.synchronize()
        assert single.shape == (250, 600)
        assert (single.cpu().numpy().astype(np.int16) ==
                oracle.canny(np.ascontiguousarray(big[2, y0:y0 + 250, x0:x0 + 600]), 1.4, 20, 60)).all()
    nchw = torch.from_numpy(np.stack([frames_of(3, 120, 200, seed=40), frames_of(3, 120, 200, seed=50)], axis=1)).cuda()
    res = torch_api.canny(nchw[:, 1], 1.4, 20, 60)
    torch.cuda.synchronize()
    host = nchw[:, 1].cpu().numpy()
    for f in range(3):
        assert (res[f].cpu().numpy().astype(np.int16) == oracle.canny(host[f], 1.4, 20, 60)).all()


def test_pitch_equal_width_is_byte_identical_to_dense(gpu_ctx):
    import torch
    n, h, w = 4, 540, 960
    d_in = torch.from_numpy(frames_of(n, h, w, seed=9)).cuda()
    a, b = torch.empty_like(d_in), torch.empty_like(d_in)
    torch.cuda.synchronize()
    cb.canny_batch_device_ptr(gpu_ctx, d_in.data_ptr(), n, h, w, 1.4, 20, 60, a.data_ptr())
    cb.canny_batch_device_strided_ptr(gpu_ctx, d_in.data_ptr(), w, h * w, n, h, w, 1.4, 20, 60, b.data_ptr(), w, h * w)
    gpu_ctx.synchronize()
    assert torch.equal(a, b)


def test_dense_and_sparse_hysteresis_strided(oracle):
    """Dense (noise) and sparse (shapes) frames alternated on one context, so both hysteresis families run on a pitched map."""
    import torch
    ctx = cb.Context(0)
    rng = np.random.default_rng(5)
    try:
        noise = frames_of(2, 270, 481, seed=21, kinds=(1,))
        shapes = frames_of(2, 270, 481, seed=22, kinds=(0,))
        for i, host in enumerate([noise, noise, shapes, shapes, noise, shapes]):
            d_in = padded_input(host, 500 + 16 * (i % 2), 1, rng)
            d_out = sentinel_output(2, 270, 499, 1)
            run_gray(ctx, d_in, d_out, 2, 270, 481, 1.4, 20, 60)
            check_result(oracle, host, d_out, 270, 481, 1.4, 20, 60, f"step {i}")
    finally:
        ctx.close()


def test_multi_chunk_with_banded_tail(gpu_ctx, oracle):
    rng = np.random.default_rng(8)
    n, h, w = 5, 1100, 640
    host = frames_of(n, h, w, seed=77)
    d_in = padded_input(host, 672, 0, rng)
    d_out = sentinel_output(n, h, 650, 1)
    gpu_ctx.set_chunk_frames(2)          # chunks of 2, 2 (the banded one) and 1 frame
    try:
        run_gray(gpu_ctx, d_in, d_out, n, h, w, 1.4, 20, 60)
    finally:
        gpu_ctx.set_chunk_frames(0)
    check_result(oracle, host, d_out, h, w, 1.4, 20, 60, "multi-chunk")


@pytest.mark.parametrize("w,in_pitch,sigma", [(640, 1920 + 64, 1.4), (640, 1920 + 5, 1.4), (644, 1932 + 16, 1.4), (640, 1920 + 64, 5.0)])
def test_bgr_fused_and_unfused(gpu_ctx, oracle, w, in_pitch, sigma):
    import torch
    from canny_edge_b200 import torch_api
    rng = np.random.default_rng(in_pitch)
    n, h = 3, 200
    bgr = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    bgr[..., 1] = frames_of(n, h, w, seed=in_pitch)    # structure in the green channel
    buf = rng.integers(0, 256, (n, h + 1, in_pitch), dtype=np.uint8)
    buf[:, :h, :3 * w] = bgr.reshape(n, h, 3 * w)
    d_buf = torch.from_numpy(buf).cuda()
    view = d_buf[:, :h, :3 * w].view(n, h, w, 3)
    out = torch.full((n, h + 1, w + 9), SENTINEL, dtype=torch.uint8, device="cuda")
    try:
        torch_api.canny_bgr(view, sigma, 20, 60, out=out[:, :h, :w], ctx=gpu_ctx)
        torch.cuda.synchronize()
    finally:
        gpu_ctx.set_stream(0)
    check_result(oracle, gray_formula(bgr), out, h, w, sigma, 20, 60, f"bgr w={w} pitch={in_pitch} sigma={sigma}")


def test_non_default_stream(oracle):
    import torch
    from canny_edge_b200 import torch_api
    host = frames_of(3, 256, 400, seed=61)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d = torch.from_numpy(host).cuda(non_blocking=False)[:, :, 8:392]
        res = torch_api.canny(d, 1.4, 20, 60)
        res2 = res.clone()                    # ordered after the edge maps on the same stream
    s.synchronize()
    for f in range(3):
        assert (res2[f].cpu().numpy().astype(np.int16) == oracle.canny(np.ascontiguousarray(host[f, :, 8:392]), 1.4, 20, 60)).all()


def test_fuzz_strided(oracle):
    import torch
    rng = np.random.default_rng(2024)
    ctx = cb.Context(0)
    tma_cases = 0
    try:
        for case in range(100):
            n = int(rng.integers(1, 4))
            h = int(rng.integers(2, 90))
            w = int(rng.integers(2, 300))
            sigma = float(rng.choice([0.5, 0.8, 1.0, 1.4, 2.0, 3.0, 5.0, 2.4]))
            lo = int(rng.integers(0, 80))
            hi = int(lo + rng.integers(-10, 100))
            # the buffer's real row stride is row = x0 + w + pad: even cases are TMA-eligible (16-byte aligned base and row), odd
            # ones mostly take the byte-load staging
            if case % 2 == 0:
                x0 = int(rng.choice([0, 16, 32]))
                row = (x0 + w + 15) // 16 * 16 + 16 * int(rng.integers(0, 2))
            else:
                x0 = int(rng.choice([0, 3, 7, 13]))
                row = x0 + w + int(rng.choice([0, 1, 5, 17]))
            in_pitch = row - x0
            tma_cases += int(x0 % 16 == 0 and row % 16 == 0)
            out_pitch = w + int(rng.choice([0, 1, 4, 7, 32]))
            host = np.empty((n, h, w), np.uint8)
            for f in range(n):
                host[f] = cb.synth_host(1, h, w, kind=int(rng.integers(0, 2)), seed=case * 10 + f)[0]
            buf = rng.integers(0, 256, (n, h + 1, in_pitch + x0), dtype=np.uint8)
            buf[:, :h, x0:x0 + w] = host
            d_buf = torch.from_numpy(buf).cuda()
            d_in = d_buf[:, :h, x0:x0 + w]
            d_out = sentinel_output(n, h, out_pitch, int(rng.integers(0, 2)))
            torch.cuda.synchronize()
            cb.canny_batch_device_strided_ptr(ctx, d_in.data_ptr(), d_in.stride(1), d_in.stride(0), n, h, w, sigma, lo, hi,
                                              d_out.data_ptr(), d_out.stride(1), d_out.stride(0))
            ctx.synchronize()
            check_result(oracle, host, d_out, h, w, sigma, lo, hi, f"case {case} n={n} {h}x{w} pitch {in_pitch}+{x0}/{out_pitch} "
                         f"sigma={sigma} {lo}/{hi}")
    finally:
        ctx.close()
    assert tma_cases >= 50, tma_cases


def test_dense_rows_with_padded_frame_stride(oracle):
    """Output rows of `width` bytes but frames padded apart: the tile-based resolve keeps its flat per-frame walk there (noise frames
    make the labelling tile-based from the second call on), the list-driven one runs for the shapes frames."""
    ctx = cb.Context(0)
    rng = np.random.default_rng(6)
    try:
        noise = frames_of(3, 200, 320, seed=31, kinds=(1,))
        shapes = frames_of(3, 200, 320, seed=32, kinds=(0,))
        for i, host in enumerate([noise, noise, noise, shapes, shapes]):
            d_in = padded_input(host, 320, 0, rng)
            d_out = sentinel_output(3, 200, 320, 5)           # pitch == width, frame stride 205 rows
            run_gray(ctx, d_in, d_out, 3, 200, 320, 1.4, 20, 60)
            check_result(oracle, host, d_out, 200, 320, 1.4, 20, 60, f"step {i}")
    finally:
        ctx.close()


def test_two_streams_without_sync(oracle):
    """Calls issued alternately on two torch streams, nothing synchronised in between: they share the cached context's workspace,
    so each must start after the previous one (b200_ctx_set_stream orders the switch).  Single-chunk and multi-chunk calls."""
    import torch
    from canny_edge_b200 import torch_api
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    hosts = [frames_of(2, 540, 960, seed=100 + 10 * i, kinds=(i % 2, 1 - i % 2)) for i in range(6)]
    hosts.append(frames_of(12, 1080, 1920, seed=200))               # 12 1080p frames: more than one chunk
    hosts.append(frames_of(12, 1080, 1920, seed=300, kinds=(1, 0)))
    d_in = [torch.from_numpy(h).cuda() for h in hosts]
    torch.cuda.synchronize()
    outs = []
    for i, d in enumerate(d_in):
        st = s1 if i % 2 == 0 else s2
        st.wait_stream(torch.cuda.default_stream())
        with torch.cuda.stream(st):
            outs.append(torch_api.canny(d[:, :, 1:], 1.4, 20, 60))
    torch.cuda.synchronize()
    for i, (h, o) in enumerate(zip(hosts, outs)):
        got = o.cpu().numpy()
        for f in range(h.shape[0]):
            want = oracle.canny(np.ascontiguousarray(h[f, :, 1:]), 1.4, 20, 60)
            assert (got[f].astype(np.int16) == want).all(), (i, f)
