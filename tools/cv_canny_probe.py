"""The OpenCV-compatible path against the reference-semantics path on one GPU, and against host cv2.Canny.

Legs, each timed with CUDA events around `--steps` calls after `--warmup` calls:
  * 512 gray 3840x2160 frames (contents: synthetic "shapes", the 256x256 test image tiled, uniform noise) through
    torch_api.cv_canny (L1 and L2, thresholds 100 / 200) and torch_api.canny (the reference's semantics, sigma 1.4, 20 / 60);
  * the same frames as 3-channel input (channels: the frame and two shifted copies) through cv_canny_color and canny_bgr;
  * one 1920x1080 gray frame per call through both paths (latency);
  * host cv2.Canny on one 4K and one 1080p frame (gray and 3-channel), for the CPU figure.
Gpix/s and the fraction of the HBM bound (7.7 TB/s at 2 B/px gray, 4 B/px 3-channel: every input byte read once, every map byte
written once).  Frame 0 of every OpenCV leg is checked against the restatement (oracle/cv_canny.py).  Prints and writes the card's
name and power limit, read in the same run, then one JSON line per leg.
    python tools/cv_canny_probe.py [--frames 512] [--steps 5] [--warmup 2] [--out profiles/r05_cv_canny_probe.jsonl]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import canny_edge_b200 as cb  # noqa: E402
from canny_edge_b200 import torch_api  # noqa: E402
from oracle.cv_canny import cv_canny as cv_oracle  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=512)
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--out", default="")
a = ap.parse_args()
N, H, W = a.frames, 2160, 3840
HBM = 7.7e12
CV_LO, CV_HI = 100.0, 200.0
SIGMA, LO, HI = 1.4, 20, 60

if not torch.cuda.is_available():
    sys.exit("cv_canny_probe: no CUDA device (GPU timings only)")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
card = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi}
print(json.dumps(card), flush=True)
results = []


def emit(r):
    results.append(r)
    print(json.dumps(r), flush=True)


def timed(fn, px):
    for _ in range(a.warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        fn()
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    return ms, px / (ms * 1e-3) / 1e9


ctx = cb.Context(0)
gray = torch.empty((N, H, W), dtype=torch.uint8, device="cuda")
out = torch.empty((N, H, W), dtype=torch.uint8, device="cuda")
test_gray = np.fromfile(ROOT / "tests" / "golden" / "test_gray_256x256.u8", dtype=np.uint8).reshape(256, 256)


def fill(content):
    if content == "test_gray_tiled":
        tile = np.tile(test_gray, (H // 256 + 1, W // 256 + 1))[:H, :W]
        gray.copy_(torch.from_numpy(tile).cuda().expand(N, H, W))
    else:
        cb.load().b200_synth_device(ctx.handle, gray.data_ptr(), N, H, W, {"shapes": 0, "noise": 1}[content], 1234, 0)
        ctx.synchronize()


def leg(name, content, fn, px, bpp, check=None):
    ms, gpix = timed(fn, px)
    bound = HBM / bpp / 1e9
    r = {"leg": name, "content": content, "frames": px // (H * W) if px >= H * W else 1, "ms_per_call": round(ms, 3),
         "gpix_s": round(gpix, 1), "hbm_bound_gpix_s": round(bound, 1), "bytes_per_px": bpp,
         "fraction_of_hbm_bound": round(gpix / bound, 4), "edge_fraction_frame0": round(float((out[0] == 255).float().mean()), 5)}
    if check is not None:
        r["frame0_equals_restatement"] = bool(check())
    emit(r)


for content in ("shapes", "test_gray_tiled", "noise"):
    fill(content)
    px = N * H * W
    host0 = gray[0].cpu().numpy()
    for l2 in (False, True):
        leg(f"cv_canny_gray_{'l2' if l2 else 'l1'}", content,
            lambda: torch_api.cv_canny(gray, CV_LO, CV_HI, L2gradient=l2, out=out, ctx=ctx), px, 2,
            check=lambda: np.array_equal(out[0].cpu().numpy(), cv_oracle(host0, CV_LO, CV_HI, l2)))
    leg("reference_canny_gray", content, lambda: torch_api.canny(gray, SIGMA, LO, HI, out=out, ctx=ctx), px, 2)
    color = torch.stack([gray, torch.roll(gray, 7, dims=2), torch.roll(gray, 5, dims=1)], dim=-1)
    host0c = color[0].cpu().numpy()
    for l2 in (False, True):
        leg(f"cv_canny_color_{'l2' if l2 else 'l1'}", content,
            lambda: torch_api.cv_canny_color(color, CV_LO, CV_HI, L2gradient=l2, out=out, ctx=ctx), px, 4,
            check=lambda: np.array_equal(out[0].cpu().numpy(), cv_oracle(host0c, CV_LO, CV_HI, l2)))
    leg("reference_canny_bgr", content, lambda: torch_api.canny_bgr(color, SIGMA, LO, HI, out=out, ctx=ctx), px, 4)
    del color
    torch.cuda.synchronize()

# one 1080p frame per call
fill("shapes")
one = gray[0, :1080, :1920].contiguous()
o1 = out[0, :1080, :1920]
for l2 in (False, True):
    leg(f"cv_canny_1080p_{'l2' if l2 else 'l1'}", "shapes", lambda: torch_api.cv_canny(one, CV_LO, CV_HI, L2gradient=l2, out=o1, ctx=ctx),
        1080 * 1920, 2)
leg("reference_canny_1080p", "shapes", lambda: torch_api.canny(one, SIGMA, LO, HI, out=o1, ctx=ctx), 1080 * 1920, 2)
torch.cuda.synchronize()
ctx.close()

# host cv2.Canny
try:
    import cv2
    for content in ("shapes", "noise"):
        fill_host = cb.synth_host(1, H, W, kind={"shapes": 0, "noise": 1}[content], seed=1234)[0]
        for (hh, ww) in ((H, W), (1080, 1920)):
            img = np.ascontiguousarray(fill_host[:hh, :ww])
            img3 = np.ascontiguousarray(np.stack([img, np.roll(img, 7, 1), np.roll(img, 5, 0)], -1))
            for name, src in (("gray", img), ("color", img3)):
                for l2 in (False, True):
                    cv2.Canny(src, CV_LO, CV_HI, L2gradient=l2)
                    reps = 5
                    t0 = time.perf_counter()
                    for _ in range(reps):
                        cv2.Canny(src, CV_LO, CV_HI, L2gradient=l2)
                    s = (time.perf_counter() - t0) / reps
                    emit({"leg": f"host_cv2_canny_{name}_{'l2' if l2 else 'l1'}", "content": content, "shape": [hh, ww],
                          "ms_per_frame": round(s * 1e3, 3), "gpix_s": round(hh * ww / s / 1e9, 3),
                          "cv2_version": cv2.__version__, "cv2_threads": cv2.getNumThreads()})
except ImportError:
    emit({"leg": "host_cv2_canny", "note": "cv2 not importable on this machine: no CPU figure"})

if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(card) + "\n")
        for r in results:
            f.write(json.dumps(r) + "\n")
