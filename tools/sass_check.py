"""SASS evidence for the front kernels (run on the CPU box; needs cuobjdump):
  * TMA (cp.async.bulk.tensor) shows up as UTMALDG, its mbarrier as SYNCS;
  * the blur's products and sums are separate multiplies and adds (FMUL2.FTZ / FADD2) — FFMA / FFMA2 only where written: the
    Markstein division steps and the exact-integer vertical Sobel;
  * opcode histogram of one instantiation, by default front3's bench kernel <R=5, TMA, DIV=1, SLAB=64, gray, dense, uniform>:
    python tools/sass_check.py > profiles/r02_front3_sass_summary.txt
"""
import collections
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
lib = ROOT / "canny_edge_b200" / "libcanny_b200.so"
want = sys.argv[1] if len(sys.argv) > 1 else "front3_kernelILi5ELb1ELi1ELi64ELb0ELb0ELb0E"
sass = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True).stdout
cur, keep = None, []
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = m.group(1)
        continue
    if cur and want in cur and re.match(r"\s+/\*[0-9a-f]{4,5}\*/", line):
        keep.append(line)
ops = collections.Counter()
for line in keep:
    t = line.split()
    op = t[2] if t[1].startswith("@") else t[1]
    ops[op.rstrip(";").split(".")[0]] += 1
print(f"# {want}: {len(keep)} SASS instructions (static), libcanny_b200.so built with -gencode arch=compute_100a,code=sm_100a")
for op, n in ops.most_common():
    print(f"{op:14s} {n}")
print()
print("UTMALDG (TMA tensor load):", ops["UTMALDG"], " SYNCS (mbarrier):", ops["SYNCS"], " FFMA2/FMUL2/FADD2 (packed fp32):",
      ops["FFMA2"] + ops["FMUL2"] + ops["FADD2"])
print("FMUL:", ops["FMUL"], " FADD:", ops["FADD"], " FFMA:", ops["FFMA"],
      "(FFMA only inside the exact division: 2 per quotient in the 3-step form, 4 in the 5-step form)")
if ops["FMUL2"] or ops["FADD2"]:
    ftz = sum(1 for line in keep if "FMUL2.FTZ" in line)
    print("packed blur: FMUL2.FTZ", ftz, "of", ops["FMUL2"], "FMUL2;  FADD2", ops["FADD2"], ";  FFMA2", ops["FFMA2"],
          "(explicit fma.rn.f32x2 only: exact division steps + the exact-integer vertical Sobel; a contracted blur would show ~400 FFMA2 and no FADD2)")
    print("half-precision Sobel: HFMA2", ops["HFMA2"], " FHFMA (fma.rn.f32.f16)", ops["FHFMA"], " F2FP", ops["F2FP"])
