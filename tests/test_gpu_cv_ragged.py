"""OpenCV-compatible frame lists on the B200 (torch_api.cv_canny_list / cv_canny_color_list, b200_cv_canny_frames_device): every map
against the numpy restatement of cv::Canny (oracle/cv_canny.py) bit for bit, and against cv2.Canny where cv2 is importable.  Inputs
sit at aligned and unaligned bases and pitches (16-byte and byte staging in one list); outputs sit in sentinel-filled buffers whose
padding must survive."""
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


def want_map(img, lo, hi, l2):
    want = cv_canny(img, lo, hi, l2)
    if cv2 is not None:
        assert np.array_equal(want, cv2.Canny(np.ascontiguousarray(img), lo, hi, L2gradient=l2)), "restatement != cv2.Canny"
    return want


def content(kind, h, w, ch, seed):
    """(h, w) or (h, w, ch) uint8: shapes, noise (every pixel a candidate at low thresholds), constant, blocks of 4 levels."""
    rng = np.random.default_rng(seed)
    if kind in ("shapes", "noise", "const"):
        k = {"shapes": 0, "noise": 1, "const": 2}[kind]
        planes = [cb.synth_host(1, h, w, kind=k, seed=seed + 17 * c)[0] for c in range(ch)]
    else:
        planes = [rng.integers(0, 256, (h, w), dtype=np.uint8) // 64 * 64 for _ in range(ch)]
    return planes[0] if ch == 1 else np.stack(planes, axis=-1)


def place(host, aligned, rng):
    """A CUDA view of `host` inside a larger buffer: base and row pitch on 16-byte boundaries (16-byte staging loads) or both odd
    (byte loads only)."""
    import torch
    h, w = host.shape[:2]
    ch = 1 if host.ndim == 2 else 3
    if aligned:
        off, pitch = 16 * int(rng.integers(0, 3)), (ch * w + 15) // 16 * 16 + 16 * int(rng.integers(0, 2))
    else:
        off, pitch = 1 + 2 * int(rng.integers(0, 8)), ch * w + 1 + 2 * int(rng.integers(0, 4))
    buf = torch.zeros(off + h * pitch + 7, dtype=torch.uint8, device="cuda")
    view = buf.as_strided((h, w) if ch == 1 else (h, w, 3), (pitch, 1) if ch == 1 else (pitch, 3, 1), off)
    view.copy_(torch.from_numpy(host))
    return view


class Outs:
    """One sentinel-filled buffer per map, the map at an offset inside it with a padded pitch."""

    def __init__(self, shapes, rng):
        import torch
        self.bufs, self.views = [], []
        for h, w in shapes:
            oy, ox = int(rng.integers(0, 3)), int(rng.integers(0, 5))
            buf = torch.full((h + oy + 1, w + ox + int(rng.integers(0, 9))), SENTINEL, dtype=torch.uint8, device="cuda")
            self.bufs.append((buf, oy, ox, h, w))
            self.views.append(buf[oy:oy + h, ox:ox + w])

    def check_padding(self, name):
        for i, (buf, oy, ox, h, w) in enumerate(self.bufs):
            pad = buf.cpu().numpy().copy()
            pad[oy:oy + h, ox:ox + w] = SENTINEL
            assert (pad == SENTINEL).all(), f"{name}: frame {i}: bytes outside its map were written"


def run_and_check(hosts, lo, hi, l2, rng, ctx=None, name="", aligned=None):
    """hosts: list of (h, w) / (h, w, 3) arrays, all of one channel count.  Returns the device views and the output views."""
    import torch
    color = hosts[0].ndim == 3
    devs = [place(x, (i % 2 == 0) if aligned is None else aligned, rng) for i, x in enumerate(hosts)]
    outs = Outs([x.shape[:2] for x in hosts], rng)
    fn = cb.torch_api.cv_canny_color_list if color else cb.torch_api.cv_canny_list
    res = fn(devs, lo, hi, L2gradient=l2, out=outs.views, ctx=ctx)
    torch.cuda.synchronize()
    assert all(r is v for r, v in zip(res, outs.views))
    for i, (x, r) in enumerate(zip(hosts, res)):
        diff = int((r.cpu().numpy() != want_map(x, lo, hi, l2)).sum())
        assert diff == 0, f"{name}: frame {i} {x.shape} (l2={l2}, {lo}, {hi}) differs in {diff} pixels"
    outs.check_padding(name)
    return devs, res


@pytest.mark.parametrize("l2", [False, True])
@pytest.mark.parametrize("ch", [1, 3])
def test_mixed_sizes(gpu_ctx, ch, l2):
    """1x1, 1xN and Nx1 up to 4K next to 256x256 in one list, contents mixed, staging forms alternating."""
    rng = np.random.default_rng(7 + ch + 10 * l2)
    sizes = [(1, 1), (2160, 3840), (1, 37), (45, 1), (256, 256), (2, 2), (3, 129), (64, 128), (67, 131), (1, 300), (300, 1),
             (130, 255), (65, 129), (1080, 1920), (5, 17)]
    kinds = ("shapes", "noise", "blocks", "const")
    hosts = [content(kinds[i % 4], h, w, ch, seed=100 + i) for i, (h, w) in enumerate(sizes)]
    run_and_check(hosts, 20, 60, l2, rng, ctx=gpu_ctx, name=f"mixed ch={ch}")
    run_and_check(hosts, 20, 60, l2, rng, ctx=gpu_ctx, name=f"mixed swapped staging ch={ch}", aligned=False)


@pytest.mark.parametrize("ch", [1, 3])
def test_test_gray_and_crops(gpu_ctx, test_gray, ch):
    """The reference's test image and crops of it at every alignment, in one list."""
    import torch
    img = test_gray if ch == 1 else np.stack([test_gray, test_gray[::-1], test_gray[:, ::-1]], axis=-1)
    big = torch.from_numpy(np.ascontiguousarray(img)).cuda()
    boxes = [(0, 256, 0, 256), (16, 200, 16, 240), (3, 250, 5, 251), (1, 2, 7, 200), (10, 200, 255, 256), (100, 101, 100, 101)]
    hosts = [np.ascontiguousarray(img[y0:y1, x0:x1]) for y0, y1, x0, x1 in boxes]
    devs = [big[y0:y1, x0:x1] for y0, y1, x0, x1 in boxes]
    fn = cb.torch_api.cv_canny_color_list if ch == 3 else cb.torch_api.cv_canny_list
    for l2 in (False, True):
        for lo, hi in ((20, 60), (100, 200), (10.5, 30.75)):
            res = fn(devs, lo, hi, L2gradient=l2, ctx=gpu_ctx)
            for i, (x, r) in enumerate(zip(hosts, res)):
                assert np.array_equal(r.cpu().numpy(), want_map(x, lo, hi, l2)), (boxes[i], l2, lo, hi)


@pytest.mark.parametrize("ch", [1, 3])
def test_mosaic_output(gpu_ctx, ch):
    """Outputs as tiles of one mosaic tensor, each tile in rows of its own at its own column; everything else must survive."""
    import torch
    rng = np.random.default_rng(3)
    sizes = [(40, 100), (1, 1), (70, 300), (1, 50), (33, 1), (64, 128), (129, 257)]
    hosts = [content(("shapes", "noise", "blocks")[i % 3], h, w, ch, seed=i) for i, (h, w) in enumerate(sizes)]
    mosaic = torch.full((sum(h for h, _ in sizes) + 3, 320), SENTINEL, dtype=torch.uint8, device="cuda")
    outs, y, placed = [], 1, []
    for i, (h, w) in enumerate(sizes):
        x = (7 * i + 3) % (320 - w + 1)
        outs.append(mosaic[y:y + h, x:x + w])
        placed.append((y, x, h, w))
        y += h
    devs = [place(x, i % 2 == 1, rng) for i, x in enumerate(hosts)]
    fn = cb.torch_api.cv_canny_color_list if ch == 3 else cb.torch_api.cv_canny_list
    fn(devs, 20, 60, out=outs, ctx=gpu_ctx)
    got = mosaic.cpu().numpy()
    rest = got.copy()
    for x, (y0, x0, h, w) in zip(hosts, placed):
        assert np.array_equal(got[y0:y0 + h, x0:x0 + w], want_map(x, 20, 60, False))
        rest[y0:y0 + h, x0:x0 + w] = SENTINEL
    assert (rest == SENTINEL).all(), "bytes of the mosaic outside the tiles were written"


@pytest.mark.parametrize("ch", [1, 3])
def test_same_input_twice(gpu_ctx, ch):
    import torch
    rng = np.random.default_rng(5)
    a = content("shapes", 150, 333, ch, seed=1)
    b = content("noise", 20, 40, ch, seed=2)
    da, db = place(a, True, rng), place(b, False, rng)
    outs = Outs([a.shape[:2], b.shape[:2], a.shape[:2], a.shape[:2]], rng)
    fn = cb.torch_api.cv_canny_color_list if ch == 3 else cb.torch_api.cv_canny_list
    fn([da, db, da, da], 20, 60, out=outs.views, ctx=gpu_ctx)
    torch.cuda.synchronize()
    wa, wb = want_map(a, 20, 60, False), want_map(b, 20, 60, False)
    for v, w in zip(outs.views, (wa, wb, wa, wa)):
        assert np.array_equal(v.cpu().numpy(), w)
    outs.check_padding("same input twice")


@pytest.mark.parametrize("l2", [False, True])
def test_multi_chunk_by_pixels(l2):
    """More than 75 Mpix: the list is cut into chunks over the three stream slots.  Every map equals the uniform call's for that
    frame alone; every third frame is also checked against the restatement."""
    import torch
    c = cb.Context(0)
    try:
        rng = np.random.default_rng(11)
        for ch in (1, 3):
            sizes = [(2160, 3840)] * 8 + [(1080, 1920), (1, 5), (777, 1001)] + [(2160, 3840)] * 4
            hosts = [content(("shapes", "noise")[i % 2], h, w, ch, seed=40 + i) for i, (h, w) in enumerate(sizes)]
            devs = [place(x, i % 3 != 1, rng) for i, x in enumerate(hosts)]
            fn = cb.torch_api.cv_canny_color_list if ch == 3 else cb.torch_api.cv_canny_list
            one = cb.torch_api.cv_canny_color if ch == 3 else cb.torch_api.cv_canny
            res = fn(devs, 30, 90, L2gradient=l2, ctx=c)
            for i, (d, r) in enumerate(zip(devs, res)):
                assert torch.equal(r, one(d, 30, 90, L2gradient=l2, ctx=c)), (ch, i)
            for i in range(0, len(hosts), 3):
                assert np.array_equal(res[i].cpu().numpy(), want_map(hosts[i], 30, 90, l2)), (ch, i)
    finally:
        c.close()


@pytest.mark.parametrize("l2", [False, True])
def test_multi_chunk_by_frame_cap(l2):
    c = cb.Context(0)
    try:
        c.set_chunk_frames(3)
        rng = np.random.default_rng(12)
        for ch in (1, 3):
            sizes = [(int(rng.integers(1, 160)), int(rng.integers(1, 260))) for _ in range(11)]
            hosts = [content(("shapes", "noise", "blocks")[i % 3], h, w, ch, seed=60 + i) for i, (h, w) in enumerate(sizes)]
            run_and_check(hosts, 20, 60, l2, rng, ctx=c, name=f"frame cap ch={ch}")
    finally:
        c.close()


@pytest.mark.parametrize("l2", [False, True])
def test_threshold_edge_cases(gpu_ctx, l2):
    rng = np.random.default_rng(21)
    for ch in (1, 3):
        hosts = [content("shapes", 150, 260, ch, seed=21), content("noise", 70, 33, ch, seed=22), content("blocks", 1, 90, ch, seed=23)]
        for lo, hi in ((0, 0), (-1, -1), (-100.5, 0.5), (60, 20), (255, 256), (2040, 2040), (2039.9, 2040.1), (1e6, 1e6), (5, 1e9),
                       (32767, 40000), (1e9, 10), (0.999, 1.001), (2.0 ** 31 - 1, 0), (-(2.0 ** 31), 100)):
            run_and_check(hosts, lo, hi, l2, rng, ctx=gpu_ctx, name=f"thresholds ch={ch}")
    import torch
    with pytest.raises(cb.CannyB200Error):   # a floor outside int32 is refused, never computed wrongly
        cb.torch_api.cv_canny_list([torch.zeros((5, 5), dtype=torch.uint8, device="cuda")], 10, 1e10, ctx=gpu_ctx)


def test_non_default_stream(gpu_ctx):
    import torch
    hosts = [content("shapes", 260, 400, 1, seed=31), content("noise", 33, 17, 1, seed=32), content("shapes", 1, 1, 1, seed=33)]
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        devs = [torch.from_numpy(x).cuda() for x in hosts]
        res = cb.torch_api.cv_canny_list(devs, 20, 60, ctx=gpu_ctx)
        res2 = cb.torch_api.cv_canny_list(devs, 20, 60, L2gradient=True, ctx=gpu_ctx)
    s.synchronize()
    for x, r, r2 in zip(hosts, res, res2):
        assert np.array_equal(r.cpu().numpy(), want_map(x, 20, 60, False))
        assert np.array_equal(r2.cpu().numpy(), want_map(x, 20, 60, True))


@pytest.mark.parametrize("ch", [1, 3])
def test_maps_equal_per_frame_cv_canny(gpu_ctx, ch):
    import torch
    rng = np.random.default_rng(77)
    sizes = [(int(rng.integers(1, 700)), int(rng.integers(1, 900))) for _ in range(40)]
    hosts = [content(("shapes", "noise", "blocks", "const")[i % 4], h, w, ch, seed=200 + i) for i, (h, w) in enumerate(sizes)]
    devs = [place(x, bool(rng.integers(0, 2)), rng) for x in hosts]
    fn = cb.torch_api.cv_canny_color_list if ch == 3 else cb.torch_api.cv_canny_list
    one = cb.torch_api.cv_canny_color if ch == 3 else cb.torch_api.cv_canny
    for l2 in (False, True):
        res = fn(devs, 25, 75, L2gradient=l2, ctx=gpu_ctx)
        for i, (d, r) in enumerate(zip(devs, res)):
            assert torch.equal(r, one(d, 25, 75, L2gradient=l2, ctx=gpu_ctx)), (i, sizes[i], l2)


def test_alternating_with_reference_semantics(gpu_ctx, oracle):
    """cv_canny_list, canny_list and the uniform cv_canny alternated on one context: the hysteresis switch is per launch, so
    canny_list's maps (with the reference's one-way link at (1,0)/(0,1)) stay equal to the reference oracle, and the OpenCV maps to
    cv::Canny."""
    import torch
    rng = np.random.default_rng(41)
    for i in range(6):
        sizes = [(int(rng.integers(2, 200)), int(rng.integers(2, 300))) for _ in range(4)]
        hosts = [content(("shapes", "noise", "blocks")[(i + k) % 3], h, w, 1, seed=50 + 10 * i + k) for k, (h, w) in enumerate(sizes)]
        devs = [torch.from_numpy(x).cuda() for x in hosts]
        l2 = bool(i & 1)
        ref = cb.torch_api.canny_list(devs, 1.4, 20, 60, ctx=gpu_ctx)
        cvl = cb.torch_api.cv_canny_list(devs, 20, 60, L2gradient=l2, ctx=gpu_ctx)
        cvu = [cb.torch_api.cv_canny(d, 20, 60, L2gradient=l2, ctx=gpu_ctx) for d in devs]
        ref2 = cb.torch_api.canny_list(devs, 1.0, 0, 30, ctx=gpu_ctx)
        torch.cuda.synchronize()
        for k, x in enumerate(hosts):
            assert np.array_equal(ref[k].cpu().numpy().astype(np.int16), oracle.canny(x, 1.4, 20, 60)), (i, k)
            assert np.array_equal(ref2[k].cpu().numpy().astype(np.int16), oracle.canny(x, 1.0, 0, 30)), (i, k)
            want = want_map(x, 20, 60, l2)
            assert np.array_equal(cvl[k].cpu().numpy(), want), (i, k)
            assert np.array_equal(cvu[k].cpu().numpy(), want), (i, k)


def test_seeded_fuzz(gpu_ctx):
    """60 seeded lists: 1-9 frames of 1..250 x 1..330, channel count, L1 / L2, staging forms, contents and thresholds at random."""
    rng = np.random.default_rng(20261021)
    for i in range(60):
        ch = int(rng.choice([1, 3]))
        n = int(rng.integers(1, 10))
        l2 = bool(rng.integers(0, 2))
        hosts = []
        for k in range(n):
            h, w = int(rng.integers(1, 251)), int(rng.integers(1, 331))
            hosts.append(content(("shapes", "noise", "const", "blocks")[int(rng.integers(0, 4))], h, w, ch, seed=1000 + 16 * i + k))
        lo, hi = float(rng.uniform(-20, 300)), float(rng.uniform(-20, 600))
        if rng.integers(0, 3) == 0:
            lo, hi = float(int(lo)), float(int(hi))
        run_and_check(hosts, lo, hi, l2, rng, ctx=gpu_ctx, name=f"fuzz {i} ch={ch} n={n}",
                      aligned=None if rng.integers(0, 2) else bool(rng.integers(0, 2)))
