#!/usr/bin/env python
"""bench.py — end-to-end Canny throughput on the BASELINE.json workloads.

Headline (config.workload): BASELINE configs[2], "batch of 512 synthetic 3840x2160 frames, sigma=1.4, frame-sharded across
1/2/4/8 B200", thresholds 20/60.  The 512 frames are the TOTAL job: rank r owns frames [r*512/N, (r+1)*512/N) — strong scaling,
no data-path collective (the frames are independent units).  A STEP is one pass of the whole hot path (blur -> Sobel/direction ->
NMS -> hysteresis) over the rank's frames.

  value         Mpix/s, whole job, inputs and outputs resident in HBM (u8 gray in, u8 0/255 edge map out).
  weak          the same with 512 frames PER GPU (round 1's headline), for the weak-scaling curve.
  e2e           same metric through the public host API (b200_canny_batch_host) with PINNED HOST buffers: H2D of every frame and D2H of
                every edge map inside the timed region; e2e.packed = b200_canny_batch_host_packed (1 bit/px maps, no host expansion).
  roofline      dominant kernel (the fused front kernel): algorithmic bytes (2 B/px: u8 in + u8 out, SURVEY 8d) per launch / its
                CUDA-event launch duration, against MEASURED_PEAKS.json's HBM copy bandwidth.  launch_ms is the kernel ALONE on the
                machine (serial re-run of the same launches on one stream); launch_ms_in_pipeline is the same launches timed inside
                the three-stream production run (they share SMs with the previous chunk's hysteresis kernels and each other's tails).
  content       device-resident Mpix/s of 64-frame batches of the three input families (shapes / tiled tests/test.jpg / noise).
  parity        GPU edge maps of the CPU sample's frames compared with the reference CPU path's, pixel by pixel.
  bgr           interleaved B,G,R frames in HBM (the reference's cvtColor step, src/main.cpp:113): converted inside the front kernel.
  latency       BASELINE configs[1]: one 1920x1080 frame, device-resident and through the host API.
  bands         BASELINE configs[4]: ONE 32768x32768 image row-band sharded over the N GPUs through the C handle (b200_bands_*):
                halo rows pulled over NVLink by the copy engines, boundary-record exchange, cross-band hysteresis merge; strong
                scaling, with a position-dependent checksum of the assembled map that must not depend on N.
  cpu_baseline  the reference's own CPU path (oracle/_ref, compiled unmodified) — or the C port when the prebuilt reference is
                absent — on a bounded sample of the same frames, on this box's cores (rank 0, N=1 only).

`--impl reference` times that CPU path instead (all host threads, bounded sample per step); it never loads the product library.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SIGMA, LO, HI = 1.4, 20, 60
ALG_BYTES_PER_PX = 2.0  # u8 gray read + u8 edge write (SURVEY 8d)
KINDS = ["shapes", "noise", "const"]
# Edge count and position-dependent checksum (b200_hash_edges_device) of the Canny map of the 32768 x 32768 "shapes" image (seed
# 1234, frame 0, sigma 1.4, 20/60).  tests/scripts/config_matrix.py compares the one-GPU map of exactly this image with the compiled
# reference (oracle/_ref, 147 s on one host thread) pixel by pixel and prints the same two numbers (profiles/r02_config_matrix.json).
BANDS_EXPECT = {(32768, 32768, 0): (16447230, "dbeef0da0fa5c89a")}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames-total", type=int, default=512, help="frames of the whole job (strong scaling: split over the GPUs)")
    ap.add_argument("--frames", type=int, default=0, help="frames PER GPU instead (weak scaling; 0 = use --frames-total)")
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--kind", type=int, default=0, help="0 shapes, 1 uniform noise, 2 constant")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-frames", type=int, default=0, help="frames in the CPU sample (0 = one per core, <= 32)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-bands", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip weak / content / latency / pipeline-profile legs")
    ap.add_argument("--workload", default="frames", choices=["frames", "bands"],
                    help="frames: the default line (with the bands object nested); bands: only the row-band run, as its own line")
    ap.add_argument("--band-height", type=int, default=32768)
    ap.add_argument("--band-width", type=int, default=32768)
    ap.add_argument("--band-steps", type=int, default=10)
    ap.add_argument("--sigma", type=float, default=SIGMA)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the edge maps of the last step (rank 0's share) to DIR/*.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs dumps the B200 arm's maps; --impl reference has none")
    return a


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


DUMP_SAMPLE_PX = 4 << 20   # float32 values + float64 indices: 48 MB, under the 64 MB a dump may take


def dump_outputs(directory, edges):
    """--dump-outputs: what the timed path returned in its last step, for comparing two builds output for output.  The inputs are
    seeded, so the same arguments give the same frames and the same sample on every run.
      edges.npy            float32 0 / 255: every pixel of the maps, or a fixed, seeded sample of DUMP_SAMPLE_PX pixels when larger
      edges_index.npy      float64: the flat C-order index of each value of edges.npy in the (frames, height, width) maps
      edges_per_frame.npy  float64: edge pixels of every frame, counted over the whole map (covers what the sample leaves out)"""
    import numpy as np
    import torch

    maps = edges.reshape(-1, edges.shape[-2], edges.shape[-1])
    flat = maps.reshape(-1)
    if flat.numel() <= DUMP_SAMPLE_PX:
        idx = np.arange(flat.numel(), dtype=np.int64)
    else:
        idx = np.unique(np.random.default_rng(1234).integers(0, flat.numel(), DUMP_SAMPLE_PX, dtype=np.int64))
    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "edges.npy", flat[torch.from_numpy(idx).to(flat.device)].float().cpu().numpy())
    np.save(out / "edges_index.npy", idx.astype(np.float64))
    np.save(out / "edges_per_frame.npy", torch.count_nonzero(maps.reshape(maps.shape[0], -1), dim=1).cpu().numpy().astype(np.float64))


# ----------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation, frame-parallel over host threads.  Nothing here touches canny_edge_b200.
# ----------------------------------------------------------------------------------------------------
def cpu_impl():
    from oracle.bindings import Oracle, Ref
    if Ref.available():
        return Ref(), "reference"
    return Oracle(), "port"


def cpu_run(frames_np, impl, threads, rounds=1, edges_out=None):
    """Runs the CPU path on every frame `rounds` times, `threads` at a time (ctypes releases the GIL). Returns wall seconds.
    edges_out: optional int16 array like frames_np that receives the maps (parity check)."""
    n = frames_np.shape[0]
    idx = iter([i % n for i in range(n * rounds)])
    lock = threading.Lock()
    is_ref = getattr(impl, "prefix", "") == "ref_"

    def work():
        while True:
            with lock:
                i = next(idx, None)
            if i is None:
                return
            if is_ref:
                out = C.c_void_p(edges_out[i].ctypes.data) if edges_out is not None else None
                impl.lib.ref_canny(C.c_void_p(frames_np[i].ctypes.data), C.c_float(SIGMA), LO, HI, frames_np.shape[1],
                                   frames_np.shape[2], out)
            else:
                e = impl.canny(frames_np[i], SIGMA, LO, HI)
                if edges_out is not None:
                    edges_out[i] = e

    ts = [threading.Thread(target=work) for _ in range(threads)]
    t0 = time.perf_counter()
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return time.perf_counter() - t0


def cpu_sample(a, n=None):
    from oracle.bindings import synth_frames
    cores = os.cpu_count() or 1
    if n is None:
        n = a.cpu_frames if a.cpu_frames > 0 else min(cores, 32)
    frames = synth_frames(n, a.height, a.width, kind=a.kind, seed=1234, first_frame=0, threads=cores)
    return frames, min(cores, n)


def run_reference(a, rank, world):
    if rank != 0:
        return
    impl, kind = cpu_impl()
    frames, threads = cpu_sample(a)
    t_one = cpu_run(frames, impl, threads)                      # first warm-up pass, also calibrates the sample
    # a step = `rounds` passes over the sample frames, sized so that the whole --warmup + --steps run stays within ~2 minutes
    rounds = max(1, min(8, int(100.0 / max(a.steps + a.warmup, 1) / max(t_one, 1e-3))))
    for _ in range(max(a.warmup - 1, 0)):
        cpu_run(frames, impl, threads, rounds)
    px = frames.size * rounds
    t = 0.0
    for _ in range(a.steps):
        t += cpu_run(frames, impl, threads, rounds)
    val = px * a.steps / t / 1e6
    sample = (f"{frames.shape[0] * rounds} frames {a.width}x{a.height} per step ({frames.shape[0]} distinct frames of the GPU arm's generator, "
              f"{rounds} passes), one frame per thread; a bounded sample of the 512-frame job (rate metric)")
    print(json.dumps({
        "impl": "reference", "metric": "end-to-end Canny Mpix/s (4K batch)", "value": round(val, 3), "unit": "Mpix/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(1e3 * t / a.steps, 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32+i16 (reference CPU arithmetic)",
        "data": "synthetic",
        "config": {"workload": f"batch of {a.width}x{a.height} synthetic frames, sigma={SIGMA}, thresholds {LO}/{HI} (BASELINE configs[2]); bounded CPU sample",
                   "frames_per_step": int(frames.shape[0] * rounds), "height": a.height, "width": a.width,
                   "generator": KINDS[a.kind] + " (oracle/canny_oracle.c::oracle_synth_rows, byte-identical to the GPU arm's)"},
        "cpu_baseline": {"value": round(val, 3), "unit": "Mpix/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": round(val, 3), "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ----------------------------------------------------------------------------------------------------
# clocks during the timed region (NVML)
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
               0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


class Env:
    """Per-process GPU state shared by the legs of the B200 arm."""

    def __init__(self, rank, world, local_rank):
        import torch
        import torch.distributed as dist

        import canny_edge_b200 as cb
        from canny_edge_b200._lib import check, load

        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference for the CPU path)")
        self.torch, self.dist, self.cb, self.check = torch, dist, cb, check
        self.rank, self.world, self.local = rank, world, local_rank
        # host placement first: this thread, the library's host pool and the pinned buffers (first touch) go to the GPU's NUMA node
        node = C.c_int(-1)
        load().b200_host_bind_numa(local_rank, C.byref(node))
        self.numa_node = node.value
        torch.cuda.set_device(local_rank)
        if world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        self.lib = load()
        self.ctx = cb.Context(local_rank)
        self.stream = torch.cuda.Stream()
        torch.cuda.set_stream(self.stream)
        self.ctx.set_stream(self.stream.cuda_stream)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([float(v)], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps, warmup):
        """warmup x fn, barrier, steps x fn between two events, barrier; returns max-over-ranks ms for the `steps` calls."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))


# ----------------------------------------------------------------------------------------------------
# GPU arm, frames
# ----------------------------------------------------------------------------------------------------
def run_b200(a, rank, world, local_rank):
    env = Env(rank, world, local_rank)
    torch, dist, cb, check, lib, ctx = env.torch, env.dist, env.cb, env.check, env.lib, env.ctx
    from canny_edge_b200 import sharded

    h, w = a.height, a.width
    weak_mode = a.frames > 0
    if weak_mode:
        first, n = rank * a.frames, a.frames
    else:
        first, n = sharded.frame_slice(a.frames_total, rank, world)
    n_total = n * world if weak_mode else a.frames_total
    n_weak = a.frames if weak_mode else a.frames_total            # frames per GPU of the weak-scaling leg
    n_buf = max(n, n_weak if not a.no_extras else n, 64)
    d_in = torch.empty((n_buf, h, w), dtype=torch.uint8, device="cuda")
    d_out = torch.empty_like(d_in)
    px = n * h * w
    check(lib.b200_synth_device(ctx.handle, d_in.data_ptr(), n, h, w, a.kind, 1234, first))
    torch.cuda.synchronize()

    def step():
        cb.canny_batch_device_ptr(ctx, d_in.data_ptr(), n, h, w, SIGMA, LO, HI, d_out.data_ptr())

    for _ in range(a.warmup):
        step()
    env.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ctx.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        step()
    e1.record()
    env.barrier()
    clocks = sampler.stop()
    launches = ctx.kernel_launches - l0
    ms = env.max_over_ranks(e0.elapsed_time(e1))
    value = n_total * h * w * a.steps / (ms * 1e-3) / 1e6
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, d_out[:n])   # before the legs below reuse d_out

    edges = C.c_ulonglong()
    check(lib.b200_count_edges_device(ctx.handle, d_out.data_ptr(), px, C.byref(edges)))

    # ---- parity against the reference CPU path on the first frames of the job (rank 0 owns frame 0...) ----
    parity = None
    cpu_frames = cpu_edges = None
    if rank == 0 and not a.no_cpu:
        impl, impl_kind = cpu_impl()
        n_par = None if world == 1 else 2          # N=1: the whole CPU sample (also timed below); N>1: two frames
        cpu_frames, cpu_threads = cpu_sample(a, n_par)
        n_par = min(cpu_frames.shape[0], n)
        import numpy as np
        cpu_edges = np.empty(cpu_frames.shape, np.int16)
        t_one = cpu_run(cpu_frames, impl, cpu_threads, 1, cpu_edges)
        got = d_out[:n_par].cpu().numpy()
        same_input = bool((d_in[:n_par].cpu().numpy() == cpu_frames[:n_par]).all())
        diff = int((got.astype(np.int16) != cpu_edges[:n_par]).sum())
        parity = {"frames_checked": int(n_par), "pixels_checked": int(n_par * h * w), "differing_pixels": diff,
                  "tolerance_band_pixels": 0, "inputs_identical": same_input, "against": impl_kind,
                  "note": "GPU map (device-resident run above) vs the CPU path on frames 0.. of the job; the blur reproduces the "
                          "reference's roundings, so the tolerance band north_star allows is empty"}

    # ---- roofline of the dominant kernel, measured live with CUDA events on the launching stream ----
    ms5, cnt5 = (C.c_float * 5)(), (C.c_int * 5)()
    check(lib.b200_profile_stages_device(ctx.handle, d_in.data_ptr(), n, h, w, C.c_float(SIGMA), LO, HI, d_out.data_ptr(), ms5, cnt5))
    # category 1 = labelling (list-driven link kernel, or tile-local union-find on dense maps), 2 = tile-border merge (dense maps
    # only), 3 = resolve (weak pixels -> 0 / 255)
    names = ["front", "hyst_label", "hyst_merge", "hyst_resolve", "other"]
    total_k = sum(ms5)
    stage = {names[i]: {"ms": round(ms5[i], 3), "launches": cnt5[i], "share": round(ms5[i] / total_k, 4) if total_k else None}
             for i in range(4)}
    peak, peak_src = peaks()
    front_launches = max(cnt5[0], 1)
    bytes_per_launch = ALG_BYTES_PER_PX * px / front_launches
    launch_ms = ms5[0] / front_launches
    achieved = bytes_per_launch / (launch_ms * 1e-3) / 1e9 if ms5[0] > 0 else 0.0
    roofline = {"bound": "hbm", "kernel": "fused front kernel (blur + Sobel + NMS + thresholds, u8 in -> u8 class map)", "achieved": round(achieved, 2),
                "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 5), "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_px": ALG_BYTES_PER_PX, "launch_ms": round(launch_ms, 4),
                "launch_ms_source": "CUDA events around every front-kernel launch of one step re-run serially on one stream (the kernel alone "
                                    "on the machine); achieved/frac use this figure",
                "front_ms_per_step_serial": round(ms5[0], 3),
                "note": "issue-bound, not HBM-bound: the reference's rounding order leaves ~34 un-fusable FP32 lane-operations per pixel for "
                        "the 11-tap separable blur alone (DESIGN.md 4.1, profiles/)",
                "whole_pipeline_frac": round(value / world * 1e6 * ALG_BYTES_PER_PX / 1e9 / peak, 5), "stages": stage}
    if not a.no_extras:
        pm5, pc5 = (C.c_float * 5)(), (C.c_int * 5)()
        check(lib.b200_profile_pipeline_device(ctx.handle, d_in.data_ptr(), n, h, w, C.c_float(SIGMA), LO, HI, d_out.data_ptr(), pm5, pc5))
        roofline["launch_ms_in_pipeline"] = round(pm5[0] / max(pc5[0], 1), 4)
        roofline["in_pipeline_note"] = ("same launches timed inside the three-stream production run: concurrent kernels share the SMs, so these "
                                        "durations overlap each other and do not add up to ms_per_step")
    prof = ROOT / "profiles" / "traffic.json"
    if prof.exists():
        try:
            t = json.loads(prof.read_text())
            per_px = t.get("front_kernel_dram_bytes_per_px")
            roofline["traffic"] = int(per_px * px / front_launches) if per_px else None
            roofline["traffic_source"] = "ncu --set full capture of one front-kernel launch (" + str(t.get("source", "profiles/")) + "), scaled per pixel to this launch size"
        except Exception:
            pass

    out = {
        "metric": "end-to-end Canny Mpix/s (4K batch)", "value": round(value, 1), "unit": "Mpix/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(ms / a.steps, 4), "higher_is_better": True,
        "scaling": "weak" if weak_mode else "strong",
        "vs_baseline": None, "dtype": "f32 blur (reference roundings) + int16/int32 gradient/NMS + u8 labels", "data": "synthetic",
        "config": {"workload": f"batch of {n_total} synthetic {w}x{h} frames, sigma={SIGMA}, thresholds {LO}/{HI}, frame-sharded over {world} GPU(s) "
                               "(BASELINE configs[2])",
                   "frames_total": n_total, "frames_per_gpu": n, "height": h, "width": w, "sigma": SIGMA, "min_val": LO, "max_val": HI,
                   "generator": KINDS[a.kind], "sharding": f"frames x{world} (no data-path collective)",
                   "l2": "inputs (%.2f GB per GPU) exceed the 126 MB L2; no flush needed" % (px / 1e9)},
        "clocks": clocks, "gpu_launches": int(launches), "edge_fraction": round(edges.value / px, 6), "roofline": roofline,
    }
    if parity:
        out["parity"] = parity

    # ---- weak scaling (512 frames per GPU) ----
    if not a.no_extras and not weak_mode:
        if world > 1:
            check(lib.b200_synth_device(ctx.handle, d_in.data_ptr(), n_weak, h, w, a.kind, 1234, rank * n_weak))
            torch.cuda.synchronize()
            wms = env.timed(lambda: cb.canny_batch_device_ptr(ctx, d_in.data_ptr(), n_weak, h, w, SIGMA, LO, HI, d_out.data_ptr()), a.steps, a.warmup)
            out["weak"] = {"value": round(world * n_weak * h * w * a.steps / (wms * 1e-3) / 1e6, 1), "unit": "Mpix/s", "frames_per_gpu": n_weak,
                           "ms_per_step": round(wms / a.steps, 4), "scaling": "weak"}
            check(lib.b200_synth_device(ctx.handle, d_in.data_ptr(), n, h, w, a.kind, 1234, first))
            torch.cuda.synchronize()
        else:
            out["weak"] = {"value": round(value, 1), "unit": "Mpix/s", "frames_per_gpu": n, "ms_per_step": round(ms / a.steps, 4), "scaling": "weak"}

    # ---- end to end through the host API: pinned host in, pinned host out ----
    if not a.no_e2e:
        # pinned host buffers for the whole per-rank batch; if the host cannot pin that much every rank falls back to the same smaller
        # number of frames
        ne = n
        while True:
            try:
                h_in = torch.empty((ne, h, w), dtype=torch.uint8, pin_memory=True)
                h_out = torch.empty((ne, h, w), dtype=torch.uint8, pin_memory=True)
                ok = 1
            except RuntimeError:
                h_in = h_out = None
                ok = 0
            if world > 1:
                t = torch.tensor([ok], device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MIN)
                ok = int(t.item())
            if ok or ne <= 8:
                break
            h_in = h_out = None
            ne //= 2
        if not ok:
            raise SystemExit("bench.py: cannot pin host memory for the e2e run")
        h_in.copy_(d_in[:ne])  # same frames as the device-resident run
        step()                 # d_out = maps of the job's frames again (the legs above reused it)
        torch.cuda.synchronize()
        px_e = ne * h * w

        def e2e_leg(fn):
            fn()
            env.barrier()
            b0h, b0d = C.c_ulonglong(), C.c_ulonglong()
            check(lib.b200_ctx_transfer_bytes(ctx.handle, C.byref(b0h), C.byref(b0d)))
            t0 = time.perf_counter()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(a.e2e_steps):
                fn()  # blocks until the last edge map is back in host memory
            g1.record()
            env.barrier()
            wall = time.perf_counter() - t0
            ems = env.max_over_ranks(max(g0.elapsed_time(g1), wall * 1e3))  # the call blocks: device timeline and host wall clock must agree
            b1h, b1d = C.c_ulonglong(), C.c_ulonglong()
            check(lib.b200_ctx_transfer_bytes(ctx.handle, C.byref(b1h), C.byref(b1d)))
            return {"value": round(world * px_e * a.e2e_steps / (ems * 1e-3) / 1e6, 1), "unit": "Mpix/s", "frames_per_gpu": ne,
                    "h2d_bytes_per_step": (b1h.value - b0h.value) // a.e2e_steps, "d2h_bytes_per_step": (b1d.value - b0d.value) // a.e2e_steps,
                    "steps": a.e2e_steps, "ms_per_step": round(ems / a.e2e_steps, 3)}

        # what the host memory system gives this rank: one pass of the library's own multi-threaded copy over the input batch
        t0 = time.perf_counter()
        h_out.copy_(h_in)
        host_copy_gbs = 2 * px_e / (time.perf_counter() - t0) / 1e9
        # ... and what PCIe gives it: plain pinned H2D copies of the same input batch (all ranks at once, like the e2e run itself)
        env.barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nce = min(ne, n_buf)
        d_in[:nce].copy_(h_in[:nce], non_blocking=True)
        c0.record()
        for _ in range(3):
            d_in[:nce].copy_(h_in[:nce], non_blocking=True)
        c1.record()
        env.barrier()
        pcie_h2d_gbs = 3 * nce * h * w / (env.max_over_ranks(c0.elapsed_time(c1)) * 1e-3) / 1e9
        e2e = e2e_leg(lambda: check(lib.b200_canny_batch_host(ctx.handle, h_in.data_ptr(), ne, h, w, C.c_float(SIGMA), LO, HI, h_out.data_ptr())))
        e2e["pcie"] = {"h2d_copy_gbs_per_gpu": round(pcie_h2d_gbs, 1), "e2e_input_gbs_per_gpu": round(e2e["value"] / world / 1e3, 1),
                       "frac_of_h2d_copy": round(e2e["value"] / world / 1e3 / pcie_h2d_gbs, 3),
                       "note": "the e2e run moves 1 B/px in (and 1/8 B/px out, the other direction): its Gpix/s per GPU against the rate of plain pinned "
                               "H2D copies of the same frames is how close the host path is to the PCIe ceiling"}
        e2e["host"] = {"numa_node_bound": env.numa_node, "pinned_copy_gbs_one_thread": round(host_copy_gbs, 1), "cpus_visible": len(os.sched_getaffinity(0)),
                       "note": "every rank's frames and maps cross the same host memory system and PCIe root complexes: the e2e figure stops scaling "
                               "where they saturate; the packed form moves 1/8 of the map bytes through host DRAM and no expansion pass"}
        e2e["api"] = ("b200_canny_batch_host (pinned host u8 frames in -> pinned host u8 0/255 edge maps out; the maps cross PCIe bit-packed and "
                      "are expanded by the library's host threads inside the timed call)")
        e2e["matches_device_run"] = bool((h_out.view(-1)[:: 4099] == d_out[:ne].cpu().view(-1)[:: 4099]).all()) if px_e < (1 << 33) else None
        if hasattr(lib, "b200_canny_batch_host_packed"):
            n_words = ne * ((h * w + 31) // 32)
            h_bits = torch.empty((n_words,), dtype=torch.int32, pin_memory=True)
            pk = e2e_leg(lambda: check(lib.b200_canny_batch_host_packed(ctx.handle, h_in.data_ptr(), ne, h, w, C.c_float(SIGMA), LO, HI, h_bits.data_ptr())))
            pk["api"] = "b200_canny_batch_host_packed (same, but the caller takes the maps as 1 bit per pixel: no host expansion pass)"
            import numpy as np
            fw = (h * w + 31) // 32                                   # words per frame
            last = ne - 1                                             # first and last frame, bit for bit
            ok_bits = True
            for f in (0, last):
                bits = np.unpackbits(h_bits.numpy()[f * fw:(f + 1) * fw].view(np.uint8), bitorder="little")[: h * w]
                ok_bits = ok_bits and bool((bits == (d_out[f].cpu().numpy().ravel() == 255)).all())
            pk["matches_device_run"] = ok_bits
            e2e["packed"] = pk
            del h_bits
        out["e2e"] = e2e
        del h_in, h_out

    # ---- other input families, 64-frame batches (device-resident) ----
    if not a.no_extras:
        import numpy as np
        nc = min(64, n_buf)
        content = {}
        for name in ("shapes", "testjpg_tiled", "noise"):
            if name == "testjpg_tiled":
                raw = ROOT / "tests" / "golden" / "test_gray_256x256.u8"
                if not raw.exists():
                    continue
                tile = torch.from_numpy(np.fromfile(raw, np.uint8).reshape(256, 256)).cuda()
                d_in[:nc] = tile.repeat(-(-h // 256), -(-w // 256))[:h, :w]
            else:
                check(lib.b200_synth_device(ctx.handle, d_in.data_ptr(), nc, h, w, 0 if name == "shapes" else 1, 1234, rank * nc))
            torch.cuda.synchronize()
            cms = env.timed(lambda: cb.canny_batch_device_ptr(ctx, d_in.data_ptr(), nc, h, w, SIGMA, LO, HI, d_out.data_ptr()), 5, 2)
            cnt = C.c_ulonglong()
            check(lib.b200_count_edges_device(ctx.handle, d_out.data_ptr(), nc * h * w, C.byref(cnt)))
            content[name] = {"value": round(world * nc * h * w * 5 / (cms * 1e-3) / 1e6, 1), "edge_fraction": round(cnt.value / (nc * h * w), 5)}
        out["content"] = {"unit": "Mpix/s", "frames_per_gpu": nc, "families": content,
                          "note": "the headline generator (shapes) is the sparsest of the three; photographs behave like testjpg_tiled"}

        # ---- interleaved B,G,R input (SURVEY 8(f)4: cvtColor(BGR2GRAY), src/main.cpp:113, folded into the front kernel's staging) ----
        if hasattr(lib, "b200_canny_batch_device_bgr") and n_buf >= 8:
            nb = min(32, n_buf // 4)
            check(lib.b200_synth_device(ctx.handle, d_in.data_ptr(), nb, h, w, 0, 1234, rank * nb))
            torch.cuda.synchronize()
            bgr = d_in[nb:4 * nb].view(nb, h, w, 3)                        # colour frames whose gray value stays close to the synthetic frame
            for ch, delta in enumerate((-9, 3, -4)):
                bgr[..., ch] = (d_in[:nb].to(torch.int16) + delta).clamp_(0, 255).to(torch.uint8)
            gray = d_out[nb:2 * nb]
            m_fused, m_gray = d_out[:nb], d_out[2 * nb:3 * nb]
            torch.cuda.synchronize()
            conv_ms = env.timed(lambda: check(lib.b200_bgr_to_gray_device(ctx.handle, bgr.data_ptr(), nb * h * w, gray.data_ptr())), 5, 2) / 5
            gms = env.timed(lambda: cb.canny_batch_device_ptr(ctx, gray.data_ptr(), nb, h, w, SIGMA, LO, HI, m_gray.data_ptr()), 5, 2) / 5
            fms = env.timed(lambda: cb.canny_batch_device_bgr_ptr(ctx, bgr.data_ptr(), nb, h, w, SIGMA, LO, HI, m_fused.data_ptr()), 5, 2) / 5
            rate = lambda ms_: round(world * nb * h * w / (ms_ * 1e-3) / 1e6, 1)
            out["bgr"] = {"unit": "Mpix/s", "frames_per_gpu": nb, "fused": rate(fms), "gray_input": rate(gms),
                          "separate_pass": rate(gms + conv_ms), "conversion_pass_alone_ms": round(conv_ms, 4),
                          "maps_equal": bool(torch.equal(m_fused, m_gray)),
                          "note": "b200_canny_batch_device_bgr: device-resident interleaved B,G,R frames; fused = converted while the front kernel "
                                  "stages its tiles (no gray plane in HBM); separate_pass = the 4 B/px conversion kernel followed by the gray "
                                  "pipeline (serial sum of the two measured times); gray values are OpenCV's fixed-point ones either way"}

        # ---- latency configuration: BASELINE configs[1], one 1920x1080 frame ----
        lh, lw = 1080, 1920
        f_in = d_in.view(-1)[: lh * lw].view(1, lh, lw)
        f_out = d_out.view(-1)[: lh * lw].view(1, lh, lw)
        check(lib.b200_synth_device(ctx.handle, f_in.data_ptr(), 1, lh, lw, 0, 1234, 0))
        torch.cuda.synchronize()
        reps = 200
        lms = env.timed(lambda: cb.canny_batch_device_ptr(ctx, f_in.data_ptr(), 1, lh, lw, SIGMA, LO, HI, f_out.data_ptr()), reps, 20)
        p_in = torch.empty((1, lh, lw), dtype=torch.uint8, pin_memory=True)
        p_out = torch.empty((1, lh, lw), dtype=torch.uint8, pin_memory=True)
        p_in.copy_(f_in)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            check(lib.b200_canny_batch_host(ctx.handle, p_in.data_ptr(), 1, lh, lw, C.c_float(SIGMA), LO, HI, p_out.data_ptr()))
        host_us = (time.perf_counter() - t0) / reps * 1e6
        out["latency"] = {"workload": "single 1920x1080 frame, sigma=1.4 (BASELINE configs[1])", "device_resident_us": round(lms / reps * 1e3, 2),
                          "pinned_host_roundtrip_us": round(host_us, 1),
                          "note": "device-resident: back-to-back calls, stream-ordered (throughput of dependent single-frame calls); host: blocking call, "
                                  "H2D + kernels + D2H"}

    del d_in, d_out
    torch.cuda.empty_cache()

    # ---- row bands of one image over the same GPUs (configs[4]) ----
    if not a.no_bands:
        out["bands"] = bands_measure(a, env, a.band_steps, a.warmup)

    # ---- CPU baseline on this box's cores (rank 0, N=1 only) ----
    if rank == 0 and world == 1 and not a.no_cpu:
        impl, kind = cpu_impl()
        threads = min(os.cpu_count() or 1, cpu_frames.shape[0])
        rounds = max(1, min(32, int(15.0 / max(t_one, 1e-3))))   # ~15 s of wall time
        secs = cpu_run(cpu_frames, impl, threads, rounds)
        out["cpu_baseline"] = {"value": round(cpu_frames.size * rounds / secs / 1e6, 3), "unit": "Mpix/s", "cores": threads, "kind": kind,
                               "sample": f"{cpu_frames.shape[0] * rounds} frames {w}x{h} ({cpu_frames.shape[0]} distinct frames of the same generator, "
                                         f"{rounds} passes), one per thread, {secs:.1f} s wall"}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------
# GPU arm, row bands of one image
# ----------------------------------------------------------------------------------------------------
def bands_measure(a, env, steps, warmup, dump=None):
    """configs[4]: one --band-height x --band-width image, row-band sharded over the GPUs; a step = halo exchange + front kernel +
    band-local labelling + boundary-record exchange + cross-band union + finalisation (b200_bands_run, csrc/bands_mgpu.cu).
    dump: directory for rank 0's band of the p2p run's last map (dump_outputs)."""
    torch, dist, check, lib, ctx = env.torch, env.dist, env.check, env.lib, env.ctx
    from canny_edge_b200 import sharded

    H, W = a.band_height, a.band_width
    rank, world = env.rank, env.world
    res = {}
    transports = ["p2p"] if world == 1 else ["p2p", "nccl"]
    for name in transports:
        os.environ["B200_BANDS_TRANSPORT"] = name
        pipe = sharded.BandPipeline(ctx, H, W, rank, world, a.sigma, LO, HI)
        g = pipe.geo
        band = pipe.band_view()   # the rank's rows live inside the handle's persistent halo buffer: no per-step copy
        edges = torch.empty((g.rows, W), dtype=torch.uint8, device="cuda")
        check(lib.b200_synth_rows_device(ctx.handle, band.data_ptr(), g.row0, g.rows, W, a.kind, 1234, 0))
        torch.cuda.synchronize()
        for _ in range(warmup):
            pipe.run(None, edges)
        env.barrier()
        pipe.timings = {}
        pipe.run(None, edges)         # one untimed step with per-stage events
        stage_ms = {k: round(v, 3) for k, v in pipe.timings.items()}
        pipe.timings = None
        env.barrier()
        l0 = ctx.kernel_launches
        sampler = ClockSampler(env.local)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            pipe.run(None, edges)
        e1.record()
        env.barrier()
        clocks = sampler.stop()
        pipe.check()
        launches = ctx.kernel_launches - l0
        ms = env.max_over_ranks(e0.elapsed_time(e1))
        if dump and rank == 0 and name == "p2p":
            dump_outputs(dump, edges)
        cnt, hsh = C.c_ulonglong(), C.c_ulonglong()
        check(lib.b200_count_edges_device(ctx.handle, edges.data_ptr(), edges.numel(), C.byref(cnt)))
        check(lib.b200_hash_edges_device(ctx.handle, edges.data_ptr(), edges.numel(), g.row0 * W, C.byref(hsh)))
        tot = torch.tensor([cnt.value, hsh.value - (1 << 64) if hsh.value >= (1 << 63) else hsh.value], device="cuda", dtype=torch.int64)
        if world > 1:
            dist.all_reduce(tot)      # int64 sums wrap: the checksum is a sum mod 2^64
        count, checksum = int(tot[0].item()), int(tot[1].item()) & ((1 << 64) - 1)
        px = H * W
        value = px * steps / (ms * 1e-3) / 1e6
        peak, peak_src = peaks()
        expect = BANDS_EXPECT.get((H, W, a.kind)) if abs(a.sigma - SIGMA) < 1e-9 else None
        r = {"value": round(value, 1), "unit": "Mpix/s", "ms_per_step": round(ms / steps, 4), "steps": steps, "scaling": "strong",
             "transport": sharded.TRANSPORTS.get(pipe.transport, str(pipe.transport)), "stage_ms_rank0": stage_ms,
             "gpu_launches": int(launches), "clocks": clocks,
             "roofline_frac_whole_pipeline": round(value * 1e6 * ALG_BYTES_PER_PX / 1e9 / world / peak, 5),
             "parity": {"edge_pixels": count, "checksum": f"{checksum:016x}",
                        "expected": ({"edge_pixels": expect[0], "checksum": expect[1]} if expect else None),
                        "matches_expected": (count == expect[0] and f"{checksum:016x}" == expect[1]) if expect else None,
                        "note": "sum over edge pixels of mix64(global pixel index) mod 2^64, all-reduced over the bands; the expected pair is the "
                                "one-GPU map's, which tests/scripts/config_matrix.py compares pixel by pixel with the compiled reference"}}
        res[name] = r
        pipe.close()
    main = res["p2p"]
    halo = sharded.band_geometry(H, W, rank, world, a.sigma).halo
    out = {"workload": f"single {W}x{H} synthetic image, sigma={a.sigma}, thresholds {LO}/{HI}, row-band sharded over {world} GPU(s) (BASELINE configs[4])",
           "height": H, "width": W, "bands": world, "band_rows": H // world, "halo_rows": halo,
           "halo_bytes_per_interior_rank_per_step": 2 * halo * W if world > 1 else 0,
           "generator": KINDS[a.kind], **main}
    if "nccl" in res:
        out["nccl_transport"] = res["nccl"]
        out["nccl_transport"]["record_bytes_all_gathered_per_step"] = world * (2 * W + 2) * 8
        out["parity"]["transports_agree"] = res["nccl"]["parity"]["checksum"] == main["parity"]["checksum"]
    return out


def run_bands(a, rank, world, local_rank):
    env = Env(rank, world, local_rank)
    b = bands_measure(a, env, a.steps, a.warmup, dump=a.dump_outputs)
    if rank == 0:
        peak, peak_src = peaks()
        print(json.dumps({
            "metric": "end-to-end Canny Mpix/s (row-band sharded image)", "value": b["value"], "unit": "Mpix/s", "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": b["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32 blur (reference roundings) + int16/int32 gradient/NMS + u8 labels", "data": "synthetic",
            "config": {k: b[k] for k in ("workload", "height", "width", "bands", "band_rows", "halo_rows", "generator", "transport")},
            "clocks": b["clocks"], "gpu_launches": b["gpu_launches"],
            "roofline": {"bound": "hbm", "kernel": "whole band pipeline", "achieved": round(b["value"] * 1e6 * ALG_BYTES_PER_PX / 1e9 / world, 2),
                         "peak": peak, "unit": "GB/s", "frac": b["roofline_frac_whole_pipeline"], "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_px": ALG_BYTES_PER_PX},
            "bands": b,
        }))
    if world > 1:
        env.dist.destroy_process_group()


def main():
    # rank 0 prints exactly one JSON line on stdout: keep NCCL's "NCCL version ..." banner (NCCL_DEBUG=VERSION/INFO) out of it
    # (VERSION and WARN both print it; with the variable unset NCCL prints nothing)
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN") and not os.environ.get("B200_KEEP_NCCL_DEBUG"):
        os.environ.pop("NCCL_DEBUG")
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank, world)
        return
    if a.workload == "bands":
        run_bands(a, rank, world, local_rank)
        return
    run_b200(a, rank, world, local_rank)


if __name__ == "__main__":
    main()
