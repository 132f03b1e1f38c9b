"""Compares two builds of libcanny_b200.so kernel by kernel (runs on the CPU box; needs cuobjdump):
  * ptxas resources (registers, stack, spills, static shared memory) from the output of `python -m canny_edge_b200.build --force -v`;
  * the `cuobjdump -sass` listing of every function, without the `identifier =` lines (the source path of each cubin) and with runs
    of blanks collapsed (cuobjdump pads its columns to the widest instruction of the cubin, which a new kernel can change).
A kernel that gained a template parameter keeps its code under a new mangled name: --rename OLD=NEW (substrings of the mangled
names) pairs the parent's kernel with the new instantiation it must still equal.
    python tools/kernel_listing_diff.py PARENT.so PARENT_BUILD.txt NEW.so NEW_BUILD.txt [--rename OLD=NEW ...] > profiles/...txt
"""
import argparse
import re
import subprocess
import sys

ap = argparse.ArgumentParser()
ap.add_argument("parent_so")
ap.add_argument("parent_log")
ap.add_argument("new_so")
ap.add_argument("new_log")
ap.add_argument("--rename", action="append", default=[])
a = ap.parse_args()
renames = [r.split("=", 1) for r in a.rename]


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, out))


def ptxas(log):
    res, cur = {}, None
    for line in open(log):
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
            res[cur] = {}
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            res[cur].update(stack=int(m.group(1)), spill=f"{m.group(2)}/{m.group(3)}")
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            sm = re.search(r"(\d+) bytes smem", line)
            res[cur].update(regs=int(m.group(1)), smem=int(sm.group(1)) if sm else 0)
            cur = None
    return {k: v for k, v in res.items() if "regs" in v}


def sass(so):
    text = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in text.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        if cur and "identifier =" not in line and line.strip():
            funcs[cur].append(" ".join(line.split()))
    return funcs


def fmt(r):
    return f"{r['regs']} regs, stack {r['stack']}, spill {r['spill']}, smem {r['smem']}" if r else "-"


def new_name(old, names):
    for o, n in renames:
        if o in old:
            cand = old.replace(o, n)
            if cand in names:
                return cand
    return old if old in names else None


pa, pb = ptxas(a.parent_log), ptxas(a.new_log)
sa, sb = sass(a.parent_so), sass(a.new_so)
names = sorted(set(pa) | set(pb))
dm = demangle(names)
same_ptx = same_sass = lines = 0
paired = set()
rows = []
for old in sorted(pa):
    new = new_name(old, pb)
    if new is None:
        rows.append((dm[old], fmt(pa[old]), "-", "gone"))
        continue
    paired.add(new)
    eq_p = pa[old] == pb[new]
    eq_s = sa.get(old) == sb.get(new)
    same_ptx += eq_p
    same_sass += eq_s
    lines += len(sa.get(old, []))
    tag = ("" if eq_p else "ptxas differs; ") + ("" if eq_s else "SASS differs")
    rows.append((dm[old] + ("" if new == old else f"  ->  {dm[new]}"), fmt(pa[old]), fmt(pb[new]), tag or "identical"))
for new in sorted(set(pb) - paired):
    rows.append((dm[new], "-", fmt(pb[new]), "new"))
print(f"# kernels: parent {len(pa)}, this change {len(pb)}; parent kernels with identical ptxas resources: {same_ptx} of {len(pa)}; "
      f"identical SASS listings: {same_sass} of {len(pa)} ({lines} SASS lines compared); new kernels: {len(set(pb) - paired)}")
w = max(len(r[0]) for r in rows)
print(f"{'kernel':{w}s}  {'parent':42s}  {'this change':42s}  result")
for r in rows:
    print(f"{r[0]:{w}s}  {r[1]:42s}  {r[2]:42s}  {r[3]}")
sys.exit(0 if same_ptx == same_sass == len(pa) else 1)
