"""cv::Canny's apertureSize 3, 5 and 7 on one GPU: for gray and 3-channel frames, L1 and L2,
  (u) 512 uniform 3840x2160 "shapes" frames through torch_api.cv_canny / cv_canny_color with apertureSize;
  (l) the seeded 2000-frame list of tools/ragged_probe.py (320x240 to 1920x1080, 16-byte and byte staging mixed) through
      cv_canny_list / cv_canny_color_list,
with thresholds 100 / 200 scaled per aperture (x1, x16, x256: magnitudes grow about 16x at 5 and 7, and 7 divides its thresholds
by 16) so that the edge density is comparable; each leg reports its edge fraction.  CUDA events around each leg after warm-up calls,
`--repeats` timed repeats; frame 0 of every leg is checked against the numpy restatement (tests/cv_canny_aperture_ref.py).  Then
per-kernel GPU times of the uniform legs (torch.profiler, CUDA activity, two calls after the warm-up), as
tools/cv_canny_kernel_times.py takes them.  Prints the card's name and power limit, then one JSON line per leg.
    python tools/cv_aperture_probe.py [--frames 512] [--list-frames 2000] [--repeats 5] [--warmup 2] [--out profiles/r08_cv_aperture_probe.jsonl]
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import canny_edge_b200 as cb  # noqa: E402
from canny_edge_b200 import torch_api  # noqa: E402
from cv_canny_aperture_ref import cv_canny as cv_ref  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=512)
ap.add_argument("--list-frames", type=int, default=2000)
ap.add_argument("--seed", type=int, default=4)
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--out", default="")
a = ap.parse_args()
T1, T2 = 100.0, 200.0
SCALE = {3: 1, 5: 16, 7: 256}
H, W = 2160, 3840

if not torch.cuda.is_available():
    sys.exit("cv_aperture_probe: no CUDA device (GPU timings only)")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
card = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi}
print(json.dumps(card), flush=True)

rng = np.random.default_rng(a.seed)   # the same draws as tools/ragged_probe.py
sizes = []
for i in range(a.list_frames):
    h, w = int(rng.integers(240, 1081)), int(rng.integers(320, 1921))
    w = w // 16 * 16 if i % 2 == 0 else w | 1        # half multiples of 16, half odd widths
    sizes.append((h, w))
list_px = sum(h * w for h, w in sizes)
uni_px = a.frames * H * W

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


def make(n, h, w, ch, frame0):
    """n "shapes" frames; channel c of a 3-channel frame is the synthetic image of seed 1234 + 17c."""
    planes = []
    for c in range(ch):
        p = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")
        lib.b200_synth_device(ctx.handle, p.data_ptr(), n, h, w, 0, 1234 + 17 * c, frame0)
        planes.append(p)
    return planes[0] if ch == 1 else torch.stack(planes, dim=-1).contiguous()


def edge_fraction(maps):
    edges = sum(int((m == 255).sum()) for m in maps)
    return round(edges / sum(m.numel() for m in maps), 5)


def matches(dev_frame, dev_map, lo, hi, l2, ap_):
    return bool(np.array_equal(dev_map.cpu().numpy(), cv_ref(dev_frame.cpu().numpy(), lo, hi, l2, ap_)))


ok = True
kernel_rows = []
for ch in (1, 3):
    one = torch_api.cv_canny_color if ch == 3 else torch_api.cv_canny
    lst = torch_api.cv_canny_color_list if ch == 3 else torch_api.cv_canny_list
    uni = make(a.frames, H, W, ch, 0)
    uout = torch.empty((a.frames, H, W), dtype=torch.uint8, device="cuda")
    frames = [make(1, h, w, ch, i)[0] for i, (h, w) in enumerate(sizes)]
    louts = [torch.empty((h, w), dtype=torch.uint8, device="cuda") for h, w in sizes]
    ctx.synchronize()
    for l2 in (False, True):
        for ap_ in (3, 5, 7):
            lo, hi = T1 * SCALE[ap_], T2 * SCALE[ap_]
            common = {"channels": ch, "l2": l2, "aperture": ap_, "thresholds": [lo, hi], "repeats": a.repeats}
            run_u = lambda: one(uni, lo, hi, apertureSize=ap_, L2gradient=l2, out=uout, ctx=ctx)   # noqa: E731
            ru = timed(run_u, uni_px)
            torch.cuda.synchronize()
            ok_u = matches(uni[0], uout[0], lo, hi, l2, ap_)
            emit({"leg": "uniform_4k", **common, "frames": a.frames, "total_mpix": round(uni_px / 1e6, 1), **ru,
                  "edge_fraction": edge_fraction([uout]), "frame0_matches_restatement": ok_u})
            rl = timed(lambda: lst(frames, lo, hi, apertureSize=ap_, L2gradient=l2, out=louts, ctx=ctx), list_px)
            torch.cuda.synchronize()
            ok_l = matches(frames[0], louts[0], lo, hi, l2, ap_)
            emit({"leg": "list_2000", **common, "frames": a.list_frames, "total_mpix": round(list_px / 1e6, 1), **rl,
                  "edge_fraction": edge_fraction(louts), "frame0_matches_restatement": ok_l})
            ok &= ok_u and ok_l
            # per-kernel GPU time of two uniform calls
            run_u()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run_u()
                run_u()
                torch.cuda.synchronize()
            kernels = {}
            for e in prof.key_averages():
                if e.device_time_total > 0 and "Memcpy" not in e.key and "Memset" not in e.key:
                    kernels[e.key.split("(")[0][:80]] = round(e.device_time_total / 1e3 / 2, 3)   # ms per call
            kernel_rows.append({"leg": "kernel_ms_per_call_uniform_4k", **common, "kernels": kernels})
            print(json.dumps(kernel_rows[-1]), flush=True)
    del uni, uout, frames, louts
    torch.cuda.empty_cache()

for ch in (1, 3):
    for leg in ("uniform_4k", "list_2000"):
        for l2 in (False, True):
            base = next(r for r in results if r["leg"] == leg and r["channels"] == ch and r["l2"] == l2 and r["aperture"] == 3)
            ratios = {f"aperture_{k}_over_3": round(next(r for r in results if r["leg"] == leg and r["channels"] == ch and
                                                         r["l2"] == l2 and r["aperture"] == k)["gpix_s"] / base["gpix_s"], 3)
                      for k in (5, 7)}
            results.append({"leg": "ratios", "of": leg, "channels": ch, "l2": l2, **ratios})
            print(json.dumps(results[-1]), flush=True)

torch.cuda.synchronize()
ctx.set_stream(0)
ctx.close()
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(card) + "\n")
        for r in results + kernel_rows:
            f.write(json.dumps(r) + "\n")
assert ok, "a map differs from the restatement"
