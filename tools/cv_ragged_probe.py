"""OpenCV-compatible frame lists on one GPU: the seeded list of tools/ragged_probe.py (frames between 320x240 and 1920x1080, half of
them with widths that are multiples of 16, so 16-byte and byte staging mix) as 1- and 3-channel frames, through
  (a) torch_api.cv_canny_list / cv_canny_color_list, one call for the whole list (and the C call alone with its frame array built once);
  (b) a Python loop of torch_api.cv_canny / cv_canny_color, one call per frame;
  (c) the same total pixels as uniform 4K frames through cv_canny / cv_canny_color,
for "shapes" and uniform-noise content (L1, thresholds 100 / 200).  Then a list of small crops (64x64, one 128x64 tile each, half
of it idle) through (a) and (b).  CUDA events around each leg after warm-up calls, `--repeats` timed repeats; the maps of (a) are
checked against those of (b).  Prints the card's name and power limit, then one JSON line per leg, channel count and content.
    python tools/cv_ragged_probe.py [--frames 2000] [--crops 20000] [--repeats 5] [--warmup 2] [--out profiles/r07_cv_ragged_probe.jsonl]
"""
import argparse
import ctypes
import json
import statistics
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import canny_edge_b200 as cb  # noqa: E402
from canny_edge_b200 import torch_api  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=2000)
ap.add_argument("--crops", type=int, default=20000)
ap.add_argument("--seed", type=int, default=4)
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--out", default="")
a = ap.parse_args()
T1, T2 = 100.0, 200.0

if not torch.cuda.is_available():
    sys.exit("cv_ragged_probe: no CUDA device (GPU timings only)")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
card = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi}
print(json.dumps(card), flush=True)

rng = np.random.default_rng(a.seed)   # the same draws as tools/ragged_probe.py
sizes = []
for i in range(a.frames):
    h, w = int(rng.integers(240, 1081)), int(rng.integers(320, 1921))
    w = w // 16 * 16 if i % 2 == 0 else w | 1        # half multiples of 16, half odd widths
    sizes.append((h, w))
total_px = sum(h * w for h, w in sizes)

ctx = cb.Context(0)
lib = cb.load()
stream = torch.cuda.Stream()
torch.cuda.set_stream(stream)
results = []


def emit(row):
    results.append(row)
    print(json.dumps(row), flush=True)


def timed(fn, px):
    for _ in range(a.warmup):
        fn()
    ms = []
    for _ in range(a.repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    med = statistics.median(ms)
    return {"ms_median": round(med, 3), "ms_min": round(min(ms), 3), "ms_max": round(max(ms), 3),
            "gpix_s": round(px / (med * 1e-3) / 1e9, 1)}


def make(h, w, ch, kind, frame):
    """One frame of content `kind`; the channels of a 3-channel frame are the synthetic images of three consecutive frame indices."""
    planes = []
    for c in range(ch):
        p = torch.empty((h, w), dtype=torch.uint8, device="cuda")
        lib.b200_synth_device(ctx.handle, p.data_ptr(), 1, h, w, kind, 1234, ch * frame + c)
        planes.append(p)
    return planes[0] if ch == 1 else torch.stack(planes, dim=-1).contiguous()


def legs(frames, ch, px):
    """(a) list call, (a') the C call alone, (b) per-frame loop; returns the three timings and whether the maps agree."""
    lst = torch_api.cv_canny_color_list if ch == 3 else torch_api.cv_canny_list
    one = torch_api.cv_canny_color if ch == 3 else torch_api.cv_canny
    out_a = [torch.empty(f.shape[:2], dtype=torch.uint8, device="cuda") for f in frames]
    out_b = [torch.empty_like(o) for o in out_a]
    ra = timed(lambda: lst(frames, T1, T2, out=out_a, ctx=ctx), px)
    arr = cb.api.frame_list([(f.data_ptr(), f.stride(0), o.data_ptr(), o.stride(0), o.shape[0], o.shape[1]) for f, o in zip(frames, out_a)])
    ra_c = timed(lambda: cb._lib.check(lib.b200_cv_canny_frames_device(ctx.handle, arr, len(frames), ch, ctypes.c_double(T1),
                                                                       ctypes.c_double(T2), 0)), px)
    rb = timed(lambda: [one(f, T1, T2, out=o, ctx=ctx) for f, o in zip(frames, out_b)], px)
    torch.cuda.synchronize()
    same = all(torch.equal(x, y) for x, y in zip(out_a, out_b))
    return ra, ra_c, rb, same


ok = True
for ch in (1, 3):
    for kind, content in ((0, "shapes"), (1, "noise")):
        frames = [make(h, w, ch, kind, i) for i, (h, w) in enumerate(sizes)]
        ctx.synchronize()
        ra, ra_c, rb, same = legs(frames, ch, total_px)
        del frames
        n4k = max(1, round(total_px / (3840 * 2160)))
        px4k = n4k * 3840 * 2160
        uni = torch.stack([make(2160, 3840, ch, kind, i) for i in range(n4k)])
        uout = torch.empty(uni.shape[:3], dtype=torch.uint8, device="cuda")
        one = torch_api.cv_canny_color if ch == 3 else torch_api.cv_canny
        rc = timed(lambda: one(uni, T1, T2, out=uout, ctx=ctx), px4k)
        del uni, uout
        common = {"channels": ch, "content": content, "frames": a.frames, "total_mpix": round(total_px / 1e6, 1), "repeats": a.repeats}
        for leg, r, extra in (("a_cv_canny_list", ra, {"maps_equal_b": same}), ("a_c_call_prebuilt_list", ra_c, {}),
                              ("b_cv_canny_loop", rb, {}), ("c_uniform_4k_cv_canny", rc, {"frames_4k": n4k})):
            emit({"leg": leg, **common, **r, **extra})
        emit({"leg": "ratios", "channels": ch, "content": content, "a_over_b": round(ra["gpix_s"] / rb["gpix_s"], 2),
              "a_over_c": round(ra["gpix_s"] / rc["gpix_s"], 3)})
        ok &= same

# small crops: every frame pays a whole 128 x 64 tile (staging, gradients, NMS of 8192 pixels for 4096)
crop_px = a.crops * 64 * 64
for ch in (1, 3):
    frames = [make(64, 64, ch, 0, i) for i in range(a.crops)]
    ctx.synchronize()
    ra, ra_c, rb, same = legs(frames, ch, crop_px)
    del frames
    common = {"channels": ch, "content": "shapes", "frames": a.crops, "size": "64x64", "total_mpix": round(crop_px / 1e6, 1),
              "repeats": a.repeats}
    for leg, r, extra in (("crops_a_cv_canny_list", ra, {"maps_equal_b": same}), ("crops_a_c_call_prebuilt_list", ra_c, {}),
                          ("crops_b_cv_canny_loop", rb, {})):
        emit({"leg": leg, **common, **r, **extra})
    emit({"leg": "crops_ratios", "channels": ch, "a_over_b": round(ra["gpix_s"] / rb["gpix_s"], 2)})
    ok &= same

torch.cuda.synchronize()
ctx.set_stream(0)
ctx.close()
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(card) + "\n")
        for r in results:
            f.write(json.dumps(r) + "\n")
assert ok, "cv_canny_list maps differ from the per-frame calls"
