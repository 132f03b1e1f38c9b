"""Builds libcanny_b200.so (hand-written sm_100a CUDA + the C ABI of include/canny_b200.h) in-tree.

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the
snapshot, so the box never needs to compile.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
LIB_PATH = PKG_DIR / "libcanny_b200.so"
SOURCES = ["front.cu", "front3.cu", "front_cv.cu", "hysteresis.cu", "stages.cu", "synth.cu", "band.cu", "bands_mgpu.cu", "selftest.cu", "api.cu"]
HEADERS = sorted(p.name for p in CSRC.glob("*.h")) + sorted(p.name for p in CSRC.glob("*.cuh")) + ["../../include/canny_b200.h"]

NVCC_FLAGS = [
    "-std=c++17", "-O3",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC",
    # no --use_fast_math / no -fmad tweaks: the blur relies on explicit __fmul_rn/__fadd_rn, the
    # division on explicit __fmaf_rn; everything else is integer.
]


# developer A/B builds: B200_NVCC_DEFS="-DF3_TAIL_IN_P1=0 ..." adds preprocessor definitions (part of the rebuild stamp)
NVCC_FLAGS += os.environ.get("B200_NVCC_DEFS", "").split()


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; libcanny_b200.so cannot be built")
    return exe


def _stamp() -> str:
    h = hashlib.sha256()
    for name in SOURCES + HEADERS:
        h.update((CSRC / name).read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> Path:
    stamp_file = PKG_DIR / ".build_stamp"
    stamp = _stamp()
    if not force and LIB_PATH.exists() and stamp_file.exists() and stamp_file.read_text() == stamp:
        return LIB_PATH
    obj_dir = PKG_DIR / "build"
    obj_dir.mkdir(exist_ok=True)
    nvcc = _nvcc()
    procs = []
    for src in SOURCES:
        obj = obj_dir / (src + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out:
            print(out)
        objs.append(str(obj))
    cmd = [nvcc, "-shared", "-o", str(LIB_PATH), *objs, "-lcudart", "-ldl"]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout)
    stamp_file.write_text(stamp)
    return LIB_PATH


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(p)
