"""Ragged frame lists on one GPU: a seeded list of frames between 320x240 and 1920x1080 (half of them with widths that are
multiples of 16, so TMA-staged and byte-staged frames mix) through
  (a) torch_api.canny_list, one call for the whole list (and the C call alone with its frame array built once);
  (b) a Python loop of torch_api.canny, one call per frame;
  (c) the same total pixels as uniform 4K frames through b200_canny_batch_device,
for "shapes" and uniform-noise content (sigma 1.4, thresholds 20 / 60).  CUDA events around each leg after warm-up calls, `--repeats`
timed repeats; the maps of (a) are checked against those of (b).  Prints the card's name and power limit, then one JSON line per
leg and content.
    python tools/ragged_probe.py [--frames 2000] [--repeats 5] [--warmup 2] [--out profiles/r04_ragged_probe.jsonl]
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
ap.add_argument("--seed", type=int, default=4)
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--out", default="")
a = ap.parse_args()
SIGMA, LO, HI = 1.4, 20, 60

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
card = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi}
print(json.dumps(card), flush=True)

rng = np.random.default_rng(a.seed)
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


for kind, content in ((0, "shapes"), (1, "noise")):
    frames = [torch.empty((h, w), dtype=torch.uint8, device="cuda") for h, w in sizes]
    for i, f in enumerate(frames):
        lib.b200_synth_device(ctx.handle, f.data_ptr(), 1, f.shape[0], f.shape[1], kind, 1234, i)
    ctx.synchronize()
    out_a = [torch.empty_like(f) for f in frames]
    out_b = [torch.empty_like(f) for f in frames]
    ra = timed(lambda: torch_api.canny_list(frames, SIGMA, LO, HI, out=out_a, ctx=ctx), total_px)
    # the C call alone, its b200_frame array built once: (a) less the Python front end's per-call work
    arr = cb.api.frame_list([(f.data_ptr(), f.stride(0), o.data_ptr(), o.stride(0), f.shape[0], f.shape[1]) for f, o in zip(frames, out_a)])
    ra_c = timed(lambda: cb._lib.check(lib.b200_canny_frames_device(ctx.handle, arr, len(frames), ctypes.c_float(SIGMA), LO, HI)),
                 total_px)
    rb = timed(lambda: [torch_api.canny(f, SIGMA, LO, HI, out=o, ctx=ctx) for f, o in zip(frames, out_b)], total_px)
    torch.cuda.synchronize()
    same = all(torch.equal(x, y) for x, y in zip(out_a, out_b))
    del frames, out_a, out_b
    n4k = max(1, round(total_px / (3840 * 2160)))
    px4k = n4k * 3840 * 2160
    uni = torch.empty((n4k, 2160, 3840), dtype=torch.uint8, device="cuda")
    lib.b200_synth_device(ctx.handle, uni.data_ptr(), n4k, 2160, 3840, kind, 1234, 0)
    ctx.synchronize()
    uout = torch.empty_like(uni)
    ctx.set_stream(stream.cuda_stream)
    rc = timed(lambda: cb.canny_batch_device_ptr(ctx, uni.data_ptr(), n4k, 2160, 3840, SIGMA, LO, HI, uout.data_ptr()), px4k)
    del uni, uout
    common = {"content": content, "frames": a.frames, "total_mpix": round(total_px / 1e6, 1), "repeats": a.repeats}
    for leg, r, extra in (("a_canny_list", ra, {"maps_equal_b": same}), ("a_c_call_prebuilt_list", ra_c, {}), ("b_canny_loop", rb, {}),
                          ("c_uniform_4k_batch", rc, {"frames_4k": n4k})):
        row = {"leg": leg, **common, **r, **extra}
        results.append(row)
        print(json.dumps(row), flush=True)
    row = {"leg": "ratios", "content": content, "a_over_b": round(ra["gpix_s"] / rb["gpix_s"], 2),
           "a_over_c": round(ra["gpix_s"] / rc["gpix_s"], 3)}
    results.append(row)
    print(json.dumps(row), flush=True)
    assert same, f"{content}: canny_list maps differ from the per-frame calls"

torch.cuda.synchronize()
ctx.set_stream(0)
ctx.close()
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(card) + "\n")
        for r in results:
            f.write(json.dumps(r) + "\n")
