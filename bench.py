#!/usr/bin/env python
"""bench.py -- headline benchmark of the GEM point-cloud -> elevation-grid fusion hot path.

Metric (BASELINE.json): Mpoints/s fused into a 1024x1024 @ 0.05 m grid, and the achieved
fraction of the HBM roofline.  One "step" = one sensor frame through the hot path:
gem_move (scroll) + gem_add_points (transform + variance + bin + per-cell Kalman fold).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N == 1 : BASELINE configs[1] (HDL-64E-shaped 10 Hz stream, 1024x1024 @ 0.05 m, 1 x B200).
N  > 1 : launched by torchrun, one rank per GPU: one sensor per rank, the global map tiled
         across ranks, points routed to their owning tile with one NCCL all-to-all
         (BASELINE configs[3]/[4] shape; weak scaling: per-GPU points fixed).
--impl reference : the reference has no CPU implementation of this path and its CUDA file
         cannot be built here (needs Eigen, SURVEY 0.3), so the reference arm times the CPU
         oracle (oracle/gem_oracle.c, a restatement of the reference semantics) on all host
         threads, kind "port".

--dump-outputs DIR (N == 1) : after the timed steps, writes the map they left behind to DIR/<layer>.npy (see
         dump_outputs); the inputs depend only on the arguments, so two builds can be compared output for output.

Prints exactly one JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALGO_BYTES_PER_POINT = 44  # SURVEY 8d: 16 B float4 in + 4 B rgba + 16 B elev/var RMW + 8 B colour/intensity write
L2_BYTES = 126e6


# ------------------------------------------------------------------------------------------
# synthetic stream
# ------------------------------------------------------------------------------------------
def _gen_one(k):
    from gem_b200 import synth
    fr = synth.hdl64_frame(k, scene=synth.make_scene())
    return k, fr


def gen_frames(nframes: int, first: int = 0):
    """frames first..first+nframes-1 of the HDL-64E stream, generated on the host cores"""
    from concurrent.futures import ProcessPoolExecutor
    workers = max(1, min(os.cpu_count() or 1, 32, nframes))
    ks = list(range(first, first + nframes))
    if workers == 1:
        out = [_gen_one(k) for k in ks]
    else:
        with ProcessPoolExecutor(workers) as ex:
            out = list(ex.map(_gen_one, ks))
    out.sort(key=lambda t: t[0])
    return [fr for _, fr in out]


def pingpong(step: int, nframes: int) -> int:
    """0,1,..,F-1,F-2,..,1,0,1,... keeps consecutive poses 1 m apart for any number of steps"""
    if nframes == 1:
        return 0
    period = 2 * nframes - 2
    r = step % period
    return r if r < nframes else period - r


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    """samples SM clock and throttle reasons of one GPU while the timed regions run"""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int = 0, period_s: float = 0.02):
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((mhz, util))
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def stop(self) -> dict:
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        mhz = [m for m, _ in self.samples]
        return {"sm_mhz": float(np.median(mhz)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(mhz)}


# ------------------------------------------------------------------------------------------
def laser_frame(fr):
    import gem_b200
    return gem_b200.make_frame(fr["T"], gem_b200.LaserSensorProcessor(), base_z=0.0)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(kernel: str):
    """per-launch DRAM bytes of the dominant kernel from the committed ncu --set full capture"""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kernel)
        except Exception:
            return None
    return None


def best_cpu_threads(frames, L: int, res: float):
    """the CPU port's best thread count on this box (persistent pool; a frame has ~0.1 ms of work per thread at 64
    threads, so the barriers start to dominate somewhere): try a few counts on a short sample and keep the best"""
    ncpu = os.cpu_count() or 1
    cands = sorted({t for t in (8, 16, 32, 48, 64, 96, ncpu) if t <= ncpu} | {min(ncpu, 8)})
    best, best_v = cands[0], -1.0
    for t in cands:
        v, _, _ = cpu_baseline(frames, 4, t, L, res, warmup=1)
        if v > best_v:
            best, best_v = t, v
    return best


def cpu_baseline(frames, nsteps: int, threads: int, L: int, res: float, warmup: int = 3):
    """CPU oracle (restatement of the reference semantics; the reference ships no CPU path) on
    `threads` host threads over the same stream.  Returns (Mpoints/s, ms/frame, n_frames)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import OracleMap
    o = OracleMap(L, res, compat_box_filter=False)
    F = len(frames)
    fobjs = [laser_frame(fr) for fr in frames]
    for s in range(warmup):  # warm-up
        k = pingpong(s, F)
        o.move(frames[k]["position"])
        o.add_pool(frames[k]["xyzi"], frames[k]["rgba"], fobjs[k], threads)
    pts = 0
    t0 = time.perf_counter()
    for s in range(nsteps):
        k = pingpong(warmup + s, F)
        o.move(frames[k]["position"])
        o.add_pool(frames[k]["xyzi"], frames[k]["rgba"], fobjs[k], threads)
        pts += frames[k]["xyzi"].shape[0]
    dt = time.perf_counter() - t0
    o.close()
    return pts / dt / 1e6, dt / nsteps * 1e3, nsteps


WORKLOAD_C2 = "configs[1]: HDL-64E-shaped synthetic 10 Hz stream into 1024x1024@0.05m robot-centric map, 1xB200"


def workload_tiled(N, L):
    return (f"{N} HDL-64E-shaped sensors (one per GPU) into one {L}x{L}@0.05m global map tiled across {N}xB200, "
            "points routed to the owning tile over NVLink (configs[3]/[4] shape)")


# ------------------------------------------------------------------------------------------
def run_reference(args):
    """Reference arm.  The reference has no CPU implementation of this path (and its CUDA file is not a CPU program),
    so this times the CPU oracle -- the restatement of the reference semantics, pinned against the reference's own
    kernels -- on the host threads, on the SAME workload as the gem_b200 arm at this --gpus value: same frame set
    (--frames distinct frames, cycled the same way), same number of warm-up and timed steps.  For N > 1 (tiled
    workload: N sensors into a (1024 N)^2 map) each step is a bounded sample: sensor 0's cloud of that step, i.e. 1/N
    of the step's points."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    N = max(1, args.gpus)
    L, res = 1024 * N, 0.05
    F = int(max(2, args.frames))
    frames = gen_frames(F)
    if N > 1:   # same rig geometry as gem_b200/tiled.py: sensor 0 of the rig, 1 m per step along +x
        from gem_b200 import tiled
        ox, oy = tiled.sensor_offset(0, N)
        for k, fr in enumerate(frames):
            T = fr["T"].copy()
            T[0, 3], T[1, 3] = ox + (k - F / 2.0), oy
            fr["T"] = T
            fr["position"] = np.array([0.0, 0.0, T[2, 3]])   # global map: no scroll
    nsteps, W = max(1, args.steps), max(0, args.warmup)
    threads = best_cpu_threads(frames[: min(F, 16)], L, res)
    o_val, ms, n = cpu_baseline(frames, nsteps, threads, L, res, warmup=W)
    ppf = float(np.mean([f["xyzi"].shape[0] for f in frames]))
    metric = "Mpoints/s fused into 1024x1024@0.05m grid" if N == 1 else "Mpoints/s fused into tiled grid"
    sample = (f"{n} frames of the c2 stream, oracle process_points+fuse, {threads} threads" if N == 1 else
              f"{n} steps, sensor 0's cloud only (1/{N} of each step's points) into the same {L}x{L} map, {threads} threads")
    line = {
        "impl": "reference", "metric": metric, "value": o_val,
        "unit": "Mpoints/s", "n_gpus": args.gpus, "steps": n, "warmup": W, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD_C2 if N == 1 else workload_tiled(N, L),
                   "points_per_frame": ppf, "distinct_frames": F, "box_filter": "off (SURVEY 8d documented deviation)",
                   "colour_path": True,
                   "note": "the reference ships no CPU path; this arm times the CPU oracle port of its semantics "
                           "(oracle/gem_oracle.c, pinned against the reference's kernels, DESIGN.md section 6)"},
        "cpu_baseline": {"value": o_val, "unit": "Mpoints/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": o_val, "unit": "Mpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    return line


def time_reference_gpu_kernels(frames, fobjs, L, res, nsteps=12):
    """extra.reference_gpu_kernels: the reference's OWN Process_points + Fuse wrappers (oracle/_ref = gpu_process.cu
    compiled unmodified against the stand-in Eigen header, with the reference's flags) on this GPU, host arrays in /
    out like the node calls them (per-call cudaMalloc/cudaMemcpy/cudaFree included: that is the reference's design).
    Wall clock per frame.  What libgem_b200 replaces."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ref_lib
    if not ref_lib.available(nofma=False):
        return {"unavailable": "oracle/_ref/libgpu_ref.so not built (needs /root/reference at build time)"}
    # the reference prints to stdout from C (gpu_process.cu:988 "GPU Init mapping"): this process' stdout carries ONE JSON line
    sys.stdout.flush()
    saved = os.dup(1)
    devnull = os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 1)
    try:
        return _time_reference_gpu_kernels(ref_lib, frames, fobjs, L, res, nsteps)
    finally:
        try:
            import ctypes
            ctypes.CDLL(None).fflush(None)   # the C library's own stdout buffer, while fd 1 still points at /dev/null
        except Exception:
            pass
        os.dup2(saved, 1)
        os.close(saved)
        os.close(devnull)


def _time_reference_gpu_kernels(ref_lib, frames, fobjs, L, res, nsteps):
    r = ref_lib.RefMap(L, res, nofma=False)
    F = len(frames)
    t_pp = t_fu = 0.0
    pts = 0
    for s in range(nsteps + 2):
        k = s % F
        fr = frames[k]
        x, y, z = (np.ascontiguousarray(fr["xyzi"][:, i]) for i in range(3))
        R, G, B = (fr["rgba"][:, i].astype(np.int32) for i in range(3))
        inten = np.ascontiguousarray(fr["xyzi"][:, 3])
        r.move(fr["position"])
        t0 = time.perf_counter()
        key, var, xt, yt, zt = r.process_points(x, y, z, fobjs[k])
        t1 = time.perf_counter()
        r.fuse_points(key, R, G, B, inten, zt, var)
        t2 = time.perf_counter()
        if s >= 2:
            t_pp += t1 - t0; t_fu += t2 - t1; pts += x.shape[0]
    return {"process_points_ms": t_pp / nsteps * 1e3, "fuse_ms": t_fu / nsteps * 1e3,
            "value": pts / (t_pp + t_fu) / 1e6, "unit": "Mpoints/s", "frames": nsteps, "grid": f"{L}x{L}@{res}",
            "what": "reference gpu_process.cu Process_points + Fuse (O(cells x points) G_fuse), host-array interface, wall clock"}


def run_c3(K=150):
    """extra.c3: BASELINE configs[2] -- D435 640x480 raw depth frames (307 200 points, NaN / out-of-range depths left
    in: the structured-light pass-through is part of the path) into a 512x512@0.02m map, frame pipeline."""
    import ctypes as C
    import torch
    import gem_b200
    from gem_b200 import synth
    dev = torch.device("cuda", 0)
    frames = [synth.d435_frame(k) for k in range(8)]
    sp = gem_b200.StructuredLightSensorProcessor()
    fobjs = [gem_b200.make_frame(fr["T"], sp, base_z=0.0) for fr in frames]
    m = gem_b200.ElevationMap(512, 0.02, compat_box_filter=False)
    st = m.torch_stream()
    xd = [torch.from_numpy(fr["xyzi"]).to(dev) for fr in frames]
    rd = [torch.from_numpy(fr["rgba"]).to(dev) for fr in frames]
    pos_c = [(C.c_float * 3)(*[float(v) for v in fr["position"]]) for fr in frames]
    n = frames[0]["xyzi"].shape[0]

    def step(s):
        k = pingpong(s, len(frames))
        m.move_fast(pos_c[k])
        m.add_stream_fast(C.c_void_p(xd[k].data_ptr()), C.c_void_p(rd[k].data_ptr()), n, C.byref(fobjs[k]))
    for s in range(20):
        step(s)
    m.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for s in range(K):
        step(20 + s)
    m.flush()
    e1.record(st)
    m.sync()
    ms = e0.elapsed_time(e1)
    stt = m.stats()
    m.close()
    return {"workload": "configs[2]: RealSense-D435 640x480 raw depth frames (307 200 points/frame, structured-light model + "
                        "depth pass-through) into 512x512@0.02m, 1xB200", "value": n * K / (ms * 1e-3) / 1e6, "unit": "Mpoints/s",
            "ms_per_step": ms / K, "frames_per_s": K / (ms * 1e-3), "last_frame_stats": stt}


def cpu_baseline_c1(threads):
    """SURVEY 8d: the CPU baseline on BASELINE configs[0] (one 64-beam frame into 200x200@0.1m)."""
    from gem_b200 import synth
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import OracleMap
    fr = synth.hdl64_frame(0)
    f = laser_frame(fr)
    out = {}
    for nt in (1, threads):
        o = OracleMap(200, 0.1, compat_box_filter=False)
        o.move(fr["position"])
        o.add_pool(fr["xyzi"], fr["rgba"], f, nt)        # warm-up (first-touch of the layers, worker creation)
        reps = 20
        t0 = time.perf_counter()
        for _ in range(reps):
            o.add_pool(fr["xyzi"], fr["rgba"], f, nt)
        dt = (time.perf_counter() - t0) / reps
        o.close()
        out[f"threads_{nt}"] = {"value": fr["xyzi"].shape[0] / dt / 1e6, "unit": "Mpoints/s", "ms_per_frame": dt * 1e3}
    out["workload"] = "configs[0]: single synthetic 64-beam frame into 200x200@0.1m, CPU oracle port (the reference has no CPU add)"
    return out


DUMP_LAYERS = ("elevation", "variance", "intensity", "color_r", "color_g", "color_b", "lowest")
DUMP_STATS = ("points_in", "points_binned", "cells_touched", "max_points_per_cell")


def dump_outputs(m, out_dir: str) -> None:
    """What a caller of gem_move + gem_add_points_stream holds after the last timed step: every layer the add path
    writes (L x L float32 each, colours converted exactly) and that step's stats (float64, DUMP_STATS order)."""
    os.makedirs(out_dir, exist_ok=True)
    m.sync()
    for name in DUMP_LAYERS:
        np.save(os.path.join(out_dir, name + ".npy"), m.get_layer(name).astype(np.float32))
    st = m.stats()
    np.save(os.path.join(out_dir, "stats.npy"), np.array([st[k] for k in DUMP_STATS], np.float64))


# ------------------------------------------------------------------------------------------
def run_single(args):
    import torch
    import gem_b200
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    L, res = 1024, 0.05
    K, W = args.steps, args.warmup
    F = int(max(2, args.frames))   # always the full set: 64 x 2.5 MB = 157 MB > L2, whatever --steps is
    frames = gen_frames(F)
    fobjs = [laser_frame(fr) for fr in frames]
    npts = [fr["xyzi"].shape[0] for fr in frames]
    in_bytes = sum(n * 20 for n in npts)
    m = gem_b200.ElevationMap(L, res, compat_box_filter=False)
    stream = m.torch_stream()   # the library-owned stream: CUDA events are recorded on it
    xyzi_d = [torch.from_numpy(fr["xyzi"]).to(dev) for fr in frames]
    rgba_d = [torch.from_numpy(fr["rgba"]).to(dev) for fr in frames]
    xyzi_h = [torch.from_numpy(fr["xyzi"]).pin_memory() for fr in frames]
    rgba_h = [torch.from_numpy(fr["rgba"]).pin_memory() for fr in frames]
    pos = [fr["position"] for fr in frames]
    flush = torch.empty(int(256e6), dtype=torch.uint8, device=dev) if in_bytes < 1.2 * L2_BYTES else None

    import ctypes as C
    pos_c = [(C.c_float * 3)(*[float(v) for v in p]) for p in pos]
    xptr = [C.c_void_p(t.data_ptr()) for t in xyzi_d]
    rptr = [C.c_void_p(t.data_ptr()) for t in rgba_d]
    xhptr = [C.c_void_p(t.data_ptr()) for t in xyzi_h]
    rhptr = [C.c_void_p(t.data_ptr()) for t in rgba_h]
    fref = [C.byref(f) for f in fobjs]

    stream_mode = os.environ.get("GEM_B200_BENCH_STREAM", "1") == "1"

    def step(s):
        k = pingpong(s, F)
        m.move_fast(pos_c[k])
        if stream_mode:    # gem_add_points_stream: consecutive frames software-pipelined
            m.add_stream_fast(xptr[k], rptr[k], npts[k], fref[k])
        else:
            m.add_fast(xptr[k], rptr[k], npts[k], fref[k])
        return npts[k]

    sampler = ClockSampler(0).start()
    # pre-populate the map (SURVEY 8d) + W untimed warm-up steps
    s0 = 0
    for s in range(10 + W):
        step(s0); s0 += 1
    torch.cuda.synchronize()

    # ---- timed region: device-resident inputs ------------------------------------------------
    m.profile_read(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pts = 0
    host_ms = None
    if flush is None:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record(stream)
        for s in range(K):
            pts += step(s0 + s)
        m.flush()                                     # the last frame's fold (deferred by the frame pipeline) is inside the timed region
        e1.record(stream)
        host_ms = (time.perf_counter() - t0) * 1e3   # time the host needed to enqueue K steps
        torch.cuda.synchronize()
        ms_total = e0.elapsed_time(e1)
    else:
        # inputs smaller than L2: flush L2 between steps and sum per-step event times
        ms_total = 0.0
        for s in range(K):
            flush.fill_(s & 255)
            torch.cuda.synchronize()
            e0.record(stream)
            pts += step(s0 + s)
            m.flush()
            e1.record(stream)
            torch.cuda.synchronize()
            ms_total += e0.elapsed_time(e1)
    launches = m.profile_read(reset=True)["launches"]
    s0 += K
    value = pts / (ms_total * 1e-3) / 1e6
    if args.dump_outputs:
        dump_outputs(m, args.dump_outputs)

    # ---- per-kernel durations: a SERIAL pass (gem_profile_enable makes the add calls issue bin -> fold_long -> fold
    # one after the other on one stream, each bracketed by CUDA events: no overlap, so the figures are uncontended) ----
    Kp = min(K, 200)
    m.profile_enable(True)
    ppts = 0
    for s in range(Kp):
        ppts += step(s0 + s)
    prof = m.profile_read(reset=True)
    m.profile_enable(False)
    s0 += Kp
    add_classes = ["bin", "fold_long", "fold", "clear_floor"]
    kname = {"bin": "k_bin", "fold_long": "k_fold_long", "fold": "k_fold", "clear_floor": "k_regions"}
    avg_us = {c: prof["ms"][c] / max(1, prof["count"][c]) * 1e3 for c in add_classes}
    dom = max(add_classes, key=lambda c: avg_us[c])
    dom_avg_ms = avg_us[dom] * 1e-3
    peak, peak_src = load_peaks()
    algo_bytes = ALGO_BYTES_PER_POINT * (ppts / Kp)
    achieved = algo_bytes / (dom_avg_ms * 1e-3) / 1e9
    tot_ms = sum(prof["ms"][c] for c in add_classes)
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": load_traffic(kname[dom]),
        "kernel": kname[dom], "kernel_avg_us": avg_us[dom], "peak_source": peak_src,
        "kernel_time_source": "serial profiling pass of this run (events around every launch, nothing overlapped); "
                              "the committed ncu launch list profiles/r2_launches_summary.txt gives the same ranking",
        "algorithmic_bytes_per_launch": algo_bytes,
        "whole_step": {"achieved": algo_bytes / (ms_total / K * 1e-3) / 1e9,
                       "frac": algo_bytes / (ms_total / K * 1e-3) / 1e9 / peak},
        "kernel_share_of_step": {kname[c]: prof["ms"][c] / max(1e-12, tot_ms) for c in add_classes},
        "kernel_us_per_launch": {kname[c]: avg_us[c] for c in add_classes},
        "note": "a c2 frame is 5.4 MB of algorithmic traffic (0.8 us at the HBM peak): the kernels are bound by dependent "
                "L2 round trips and the serial fold of the longest per-cell list, not by bandwidth (DESIGN.md section 4)",
    }

    # ---- e2e: host (pinned) buffers through the public API, H2D + D2H inside the timed region ------
    Ke = K
    for s in range(min(W, 5)):
        k = pingpong(s0, F); m.move(pos[k]); m.add(xyzi_h[k].numpy(), rgba_h[k].numpy(), fobjs[k]); s0 += 1
    torch.cuda.synchronize()
    epts = 0
    t0 = time.perf_counter()
    e0.record(stream)
    for s in range(Ke):
        k = pingpong(s0 + s, F)
        m.move_fast(pos_c[k])
        m.add_host_fast(xhptr[k], rhptr[k], npts[k], fref[k])   # H2D 20 B/pt, kernels, D2H counters, sync
        epts += npts[k]
    e1.record(stream)
    torch.cuda.synchronize()
    e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    s0 += Ke
    e2e_sync_value = epts / (e2e_ms * 1e-3) / 1e6
    # pipelined variant of the same public call: H2D of frame i+1 overlaps the kernels of frame i
    # (three staging buffers, copy stream); every step still does its own H2D and a counters D2H
    for s in range(4):
        k = pingpong(s0, F); m.move_fast(pos_c[k]); m.add_host_async_fast(xhptr[k], rhptr[k], npts[k], fref[k]); s0 += 1
    m.sync()
    torch.cuda.synchronize()
    apts = 0
    t0 = time.perf_counter()
    e0.record(stream)
    for s in range(Ke):
        k = pingpong(s0 + s, F)
        m.move_fast(pos_c[k])
        m.add_host_async_fast(xhptr[k], rhptr[k], npts[k], fref[k])
        apts += npts[k]
    m.flush()
    e1.record(stream)
    m.sync()
    torch.cuda.synchronize()
    a_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    s0 += Ke
    ctr_bytes = 768
    e2e = {"value": apts / (a_ms * 1e-3) / 1e6, "unit": "Mpoints/s",
           "h2d_bytes_per_step": 20.0 * apts / Ke, "d2h_bytes_per_step": ctr_bytes,
           "api": "gem_move + gem_add_points_host_async (pinned host xyzi+rgba in via copy stream, counters out; "
                  "wall clock incl. final sync)",
           "host_synchronous_variant": {"value": e2e_sync_value, "api": "gem_move + gem_add_points_host (sync per frame)"}}

    # ---- e2e_frame: what a node waits for per sensor frame, through the public calls, from 32-byte PCL records in
    # pinned host memory: Move + add (gem_add_cloud_pcl_host: H2D + bin + fold) + Mapvar_update + Map_feature's kernel
    # + grid_map write-back (9 layers into pinned host memory) + Raytracing ----
    Kf = min(K, 30)
    pcl_h = []
    for fr in frames[: min(F, 8)]:
        rec = np.zeros((fr["xyzi"].shape[0], 8), np.float32)
        rec[:, :3] = fr["xyzi"][:, :3]; rec[:, 3] = 1.0
        bgra = np.stack([fr["rgba"][:, 2], fr["rgba"][:, 1], fr["rgba"][:, 0], np.full(fr["rgba"].shape[0], 255, np.uint8)], 1)
        rec[:, 4] = np.ascontiguousarray(bgra).view(np.float32).reshape(-1)
        rec[:, 6] = fr["xyzi"][:, 3]
        pcl_h.append(torch.from_numpy(rec).pin_memory())
    ex_pin = {n: torch.empty((L, L), dtype=torch.float32).pin_memory() for n in gem_b200._lib.EXPORT_LAYERS}
    ex = {n: ex_pin[n].numpy().T for n in ex_pin}   # column-major views of pinned host memory
    for s in range(3):
        k = pingpong(s0 + s, F) % len(pcl_h)
        m.move(pos[k]); m.add_pcl(pcl_h[k].numpy(), fobjs[k]); m.var_update(0.0); m.compute_features(); m.export_layers(ex); m.raytracing()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s in range(Kf):
        k = pingpong(s0 + 3 + s, F) % len(pcl_h)
        m.move(pos[k]); m.add_pcl(pcl_h[k].numpy(), fobjs[k])
        m.var_update(0.0); m.compute_features(); m.export_layers(ex); m.raytracing()
    torch.cuda.synchronize()
    frame_ms = (time.perf_counter() - t0) * 1e3 / Kf
    # the same frame with the write-back overlapped with the ray clean-up (gem_export_layers_begin / _end), for all nine
    # layers and for the three a planner reads (elevation, variance, traversability)
    overlapped = {}
    for label, names in (("nine_layers", None), ("three_layers", ["elevation", "variance", "traver"])):
        t0 = time.perf_counter()
        for s in range(Kf):
            k = pingpong(s0 + 3 + s, F) % len(pcl_h)
            m.move(pos[k]); m.add_pcl(pcl_h[k].numpy(), fobjs[k])
            m.var_update(0.0); m.compute_features(); m.export_layers_begin(ex, names); m.raytracing(); m.export_layers_end()
        torch.cuda.synchronize()
        overlapped[label] = (time.perf_counter() - t0) * 1e3 / Kf
    e2e_frame = {"ms_per_frame": frame_ms, "frames": Kf, "ms_per_frame_export_overlapped": overlapped,
                 "api": "gem_move + gem_add_cloud_pcl_host (32 B PointXYZRGBICT records from pinned host memory) + gem_var_update + "
                        "gem_compute_features + gem_export_layers (9 column-major layers into pinned host memory) + gem_raytracing, "
                        "host-synchronous like the node",
                 "h2d_bytes_per_frame": 32.0 * float(np.mean(npts)), "d2h_bytes_per_frame": 9 * 4 * L * L}
    clocks = sampler.stop()

    # ---- secondary: BASELINE configs[4] shape on ONE GPU: 8 sensors x ~123 k points per launch into an
    # 8192x8192 @ 0.05 m map through gem_add_points_multi (launch latency and the fold tail amortised) -----
    extra = {}
    for name, fn in (("c5_shape_one_gpu", lambda: run_multi_sensor(frames, fobjs, npts, peak)), ("c3", run_c3),
                     ("reference_gpu_kernels_c2", lambda: time_reference_gpu_kernels(frames[:8], fobjs[:8], 1024, 0.05)),
                     ("reference_gpu_kernels_c1", lambda: time_reference_gpu_kernels(frames[:4], fobjs[:4], 200, 0.1))):
        try:
            extra[name] = fn()
        except Exception as e:  # never let a secondary measurement break the headline line
            extra[name] = {"error": repr(e)}

    # ---- the tiled path at world = 1 (what `--gpus N` times, on one GPU): the baseline its scaling curve is read against ----
    try:
        import subprocess
        env = dict(os.environ, GEM_B200_BENCH_PARITY="0", MASTER_ADDR="127.0.0.1")
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=1", "--master-addr", "127.0.0.1",
                            "--master-port", "29677", os.path.abspath(__file__), "--gpus", "2", "--steps", str(min(K, 400)), "--warmup", "10",
                            "--frames", str(min(F, 32))], capture_output=True, text=True, timeout=240, env=env)
        tl = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        extra["tiled_path_world1"] = {"value": tl["value"], "unit": "Mpoints/s", "ms_per_step": tl["ms_per_step"],
                                      "what": "bench.py --gpus N's code path (gem_tiled_step: route + peer bin + fold, pipelined) with one rank that "
                                              "owns the whole 1024x1024 map; the N-GPU lines divide by N times THIS for the tiled path's own efficiency"}
    except Exception as e:
        extra["tiled_path_world1"] = {"error": repr(e)}

    # ---- CPU baseline beside it (bounded sample) ----------------------------------------------------
    threads = best_cpu_threads(frames[: min(F, 16)], L, res)
    nb = int(min(max(K, 5), 40))
    cb_val, cb_ms, cb_n = cpu_baseline(frames[: min(F, 16)], nb, threads, L, res)
    cb1_val, _, _ = cpu_baseline(frames[: min(F, 16)], min(nb, 10), 1, L, res)
    try:
        extra["cpu_baseline_c1"] = cpu_baseline_c1(threads)
    except Exception as e:
        extra["cpu_baseline_c1"] = {"error": repr(e)}

    st = m.stats()
    extra.update({"host_enqueue_ms_per_step": (host_ms / K) if host_ms is not None else None,
                  "e2e_frame": e2e_frame, "last_frame_stats": st, "host_cores": os.cpu_count()})
    line = {
        "metric": "Mpoints/s fused into 1024x1024@0.05m grid", "value": value, "unit": "Mpoints/s", "n_gpus": 1,
        "steps": K, "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD_C2,
                   "step": ("gem_move + gem_add_points_stream on one frame (device-resident float4 xyzi + uchar4 rgba; "
                            "consecutive frames software-pipelined: one CUDA graph {fold of frame i-1 || bin of frame i} per call)"
                            if stream_mode else "gem_move + gem_add_points on one frame (device-resident float4 xyzi + uchar4 rgba)"),
                   "points_per_frame": float(np.mean(npts)), "distinct_frames": F,
                   "l2": (f"inputs larger than L2: {F} distinct frames = {in_bytes/1e6:.0f} MB cycled" if flush is None
                          else "L2 flushed (256 MB write) between timed steps"),
                   "box_filter": "off (SURVEY 8d documented deviation)", "colour_path": True},
        "roofline": roofline,
        "cpu_baseline": {"value": cb_val, "unit": "Mpoints/s", "cores": threads, "kind": "port",
                         "sample": f"{cb_n} frames of the same stream, oracle process_points+fuse on {threads} threads; "
                                   f"single thread: {cb1_val:.1f} Mpoints/s", "single_thread_value": cb1_val},
        "e2e": e2e, "clocks": clocks, "gpu_launches": int(launches),
        "extra": extra,
    }
    return line


def run_multi_sensor(frames, fobjs, npts, peak, nsens=8, K=200):
    import torch
    import gem_b200
    from gem_b200 import tiled
    dev = torch.device("cuda", 0)
    L, res = 8192, 0.05
    m = gem_b200.ElevationMap(L, res, compat_box_filter=False, max_points=1 << 21)
    stream = m.torch_stream()
    F = len(frames)
    nsets = min(16, F // nsens * 2) or 1
    sets = []
    for sidx in range(nsets):
        ks = [(sidx * 3 + j * 5) % F for j in range(nsens)]
        x = torch.from_numpy(np.concatenate([frames[k]["xyzi"] for k in ks])).to(dev)
        c = torch.from_numpy(np.concatenate([frames[k]["rgba"] for k in ks])).to(dev)
        off = np.concatenate([[0], np.cumsum([npts[k] for k in ks])])
        fr = []
        for j, k in enumerate(ks):
            ox, oy = tiled.sensor_offset(j, nsens)
            T = frames[k]["T"].copy()
            T[0, 3] = ox + (sidx - nsets / 2.0)
            T[1, 3] = oy
            fr.append(gem_b200.make_frame(T, gem_b200.LaserSensorProcessor()))
        sets.append((x, c, off, fr, int(off[-1])))
    for s in range(12):
        x, c, off, fr, n = sets[s % nsets]
        m.add_multi(x, c, off, fr)
    m.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pts = 0
    e0.record(stream)
    for s in range(K):
        x, c, off, fr, n = sets[s % nsets]
        m.add_multi(x, c, off, fr)
        pts += n
    e1.record(stream)
    m.sync()
    ms = e0.elapsed_time(e1)
    m.profile_enable(True)
    for s in range(50):
        x, c, off, fr, n = sets[s % nsets]
        m.add_multi(x, c, off, fr)
    pr = m.profile_read(reset=True)
    st = m.stats()
    m.close()
    gbs = ALGO_BYTES_PER_POINT * pts / (ms * 1e-3) / 1e9
    return {"workload": f"{nsens} HDL-64E-shaped sensors per launch (gem_add_points_multi) into 8192x8192@0.05m, 1xB200",
            "value": pts / (ms * 1e-3) / 1e6, "unit": "Mpoints/s", "ms_per_step": ms / K, "points_per_step": pts / K,
            "achieved_GBps_algorithmic": gbs, "frac_of_hbm_peak": gbs / peak,
            "kernel_us_per_step": {k: v / 50 * 1e3 for k, v in pr["ms"].items() if v}, "last_step_stats": st}


# ------------------------------------------------------------------------------------------
def run_tiled(args):
    from gem_b200 import tiled
    return tiled.bench(args, gen_frames, pingpong, laser_frame, ClockSampler, load_peaks, ALGO_BYTES_PER_POINT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="gem_b200", choices=["gem_b200", "reference"])
    ap.add_argument("--frames", type=int, default=64, help="distinct synthetic frames cycled (64 x 2.5 MB > L2)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the map the timed steps left behind to DIR/<layer>.npy (--gpus 1 only)")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl != "gem_b200" or args.gpus > 1 or world > 1):
        ap.error("--dump-outputs is supported on the single-GPU gem_b200 path only")
    if args.impl == "reference":
        line = run_reference(args)
    elif args.gpus > 1 or world > 1:
        line = run_tiled(args)
    else:
        line = run_single(args)
    if line is not None:
        print(json.dumps(line))


if __name__ == "__main__":
    main()
