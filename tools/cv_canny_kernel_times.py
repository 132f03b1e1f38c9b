"""Per-kernel GPU time of the OpenCV-compatible path and of the reference-semantics path on the same 512 synthetic 4K "shapes"
frames (torch.profiler, CUDA activity), two calls each after two warm-up calls.  Kernels of the three stream slots overlap, so the
sums exceed the wall time of a call.
    python tools/cv_canny_kernel_times.py [--out profiles/r05_cv_kernel_times.txt]
"""
import argparse
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import canny_edge_b200 as cb  # noqa: E402
from canny_edge_b200 import torch_api  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="")
a = ap.parse_args()
N, H, W = 512, 2160, 3840
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
lines = [f"# {torch.cuda.get_device_name(0)} ({smi}); 512 x 3840x2160 shapes frames, two calls per table"]
ctx = cb.Context(0)
g = torch.empty((N, H, W), dtype=torch.uint8, device="cuda")
o = torch.empty_like(g)
cb.load().b200_synth_device(ctx.handle, g.data_ptr(), N, H, W, 0, 1234, 0)
ctx.synchronize()
for name, fn in (("cv_canny L1, thresholds 100 / 200", lambda: torch_api.cv_canny(g, 100, 200, out=o, ctx=ctx)),
                 ("canny (reference semantics), sigma 1.4, 20 / 60", lambda: torch_api.canny(g, 1.4, 20, 60, out=o, ctx=ctx))):
    fn()
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        fn()
        fn()
        torch.cuda.synchronize()
    lines.append(f"== {name}")
    lines.append(p.key_averages().table(sort_by="cuda_time_total", row_limit=4, max_name_column_width=60))
ctx.close()
text = "\n".join(lines)
print(text)
if a.out:
    Path(a.out).write_text(text + "\n")
