"""Strided device batches against the contiguous call on one GPU: Gpix/s of the same synthetic 4K "shapes" frames (sigma 1.4,
thresholds 20 / 60) through every staging form the strided entry points have, plus what a caller pays today for a crop (a
.contiguous() copy, then the contiguous call).  CUDA events around `--steps` calls after `--warmup` calls of each leg; every leg's
maps are checked against the contiguous call's.  Prints the card's name and power limit, then one JSON line per leg.
    python tools/strided_probe.py [--frames 512] [--steps 5] [--warmup 2] [--out profiles/r03_strided_probe.jsonl]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch  # noqa: E402

import canny_edge_b200 as cb  # noqa: E402
from canny_edge_b200 import torch_api  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=512)
ap.add_argument("--height", type=int, default=2160)
ap.add_argument("--width", type=int, default=3840)
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--out", default="")
a = ap.parse_args()
n, h, w = a.frames, a.height, a.width
SIGMA, LO, HI = 1.4, 20, 60

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
card = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi}
print(json.dumps(card), flush=True)

ctx = cb.Context(0)
gray = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")
cb.load().b200_synth_device(ctx.handle, gray.data_ptr(), n, h, w, 0, 1234, 0)
ctx.synchronize()
ref = torch.empty_like(gray)
stream = torch.cuda.Stream()
torch.cuda.set_stream(stream)
ctx.set_stream(stream.cuda_stream)


def timed(fn):
    for _ in range(a.warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        fn()
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    return ms, n * h * w / (ms * 1e-3) / 1e9


results = []


def leg(name, fn, out_view, detail):
    ms, gpix = timed(fn)
    same = bool(torch.equal(out_view, ref))
    r = {"leg": name, "ms_per_call": round(ms, 3), "gpix_s": round(gpix, 1), "maps_equal_contiguous": same, **detail}
    results.append(r)
    print(json.dumps(r), flush=True)


# 1. the existing contiguous call
timed(lambda: cb.canny_batch_device_ptr(ctx, gray.data_ptr(), n, h, w, SIGMA, LO, HI, ref.data_ptr()))
out = torch.empty_like(gray)
leg("contiguous", lambda: cb.canny_batch_device_ptr(ctx, gray.data_ptr(), n, h, w, SIGMA, LO, HI, out.data_ptr()), out,
    {"pitch": w})
# 2. the strided call with pitch = width
leg("strided_pitch_eq_width", lambda: cb.canny_batch_device_strided_ptr(ctx, gray.data_ptr(), w, h * w, n, h, w, SIGMA, LO, HI,
                                                                         out.data_ptr(), w, h * w), out, {"pitch": w})
del out
# 3. padded pitch of 4096 for input and output (TMA staging)
pin = torch.zeros((n, h, 4096), dtype=torch.uint8, device="cuda")
pin[:, :, :w] = gray
pout = torch.zeros((n, h, 4096), dtype=torch.uint8, device="cuda")
leg("padded_pitch_4096", lambda: torch_api.canny(pin[:, :, :w], SIGMA, LO, HI, out=pout[:, :, :w], ctx=ctx), pout[:, :, :w],
    {"pitch": 4096, "staging": "tma"})
del pin, pout
# 4. a crop at an unaligned column offset (byte-load staging), output dense
x0 = 3
src = torch.zeros((n, h, w + 16), dtype=torch.uint8, device="cuda")
src[:, :, x0:x0 + w] = gray
crop = src[:, :, x0:x0 + w]
out = torch.empty_like(gray)
leg("crop_unaligned_x3", lambda: torch_api.canny(crop, SIGMA, LO, HI, out=out, ctx=ctx), out,
    {"pitch": w + 16, "column_offset": x0, "staging": "byte loads"})
# 5. the same crop made contiguous first, then the contiguous call (the copy is inside the timed window)
def copy_then_contiguous_call():
    dense = crop.contiguous()
    cb.canny_batch_device_ptr(ctx, dense.data_ptr(), n, h, w, SIGMA, LO, HI, out.data_ptr())


ctx.set_stream(stream.cuda_stream)
leg("crop_contiguous_copy", copy_then_contiguous_call, out,
    {"pitch": w, "column_offset": x0, "note": ".contiguous() copy + b200_canny_batch_device"})
del src, crop
# 6. / 7. B,G,R frames whose gray value is the synthetic frame's (B = G = R = g), padded pitches
for name, pitch, detail in (("bgr_padded_pitch", 3 * w + 64, {"conversion": "fused"}),
                            ("bgr_unaligned_pitch", 3 * w + 5, {"conversion": "separate strided pass"})):
    buf = torch.zeros((n, h, pitch), dtype=torch.uint8, device="cuda")
    view = buf[:, :, :3 * w].view(n, h, w, 3)
    view.copy_(gray.unsqueeze(-1).expand(n, h, w, 3))
    leg(name, lambda: torch_api.canny_bgr(view, SIGMA, LO, HI, out=out, ctx=ctx), out, {"pitch": pitch, **detail})
    del buf, view
torch.cuda.synchronize()
ctx.set_stream(0)
ctx.close()
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(card) + "\n")
        for r in results:
            f.write(json.dumps(r) + "\n")
