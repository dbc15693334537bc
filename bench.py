#!/usr/bin/env python
"""Benchmark of the warp-and-fuse hot path (BASELINE.json metric: SR frames/s, 4x, 1080p out; projection+warp
GB/s vs HBM peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload, identical in both arms) = configs[1] "C2": 4x VSR 480x270 -> 1920x1080, 7-frame window
(M = 20 stacked maps), batch 1 per GPU.  One step = one output frame through WarpFusePipeline.step: 6 flow projections,
6 depth-aware projections, the chained centre->neighbour flows, 6 bilinear warps (+ fused residual norm), mask
threshold + label warp, stack assembly, and the fusion conv stack twice (pass 1 + fuse pass,
network/video_super_resolution.py:41,64).  At N > 1 every rank runs its own window (weak scaling, no collective on
the hot path); the u8 output frames are all-gathered once after the last step (NCCL), inside the timed region.

One JSON line on stdout (rank 0):
  value     frames/s with inputs resident in HBM
  e2e       frames/s through the public API with pinned HOST inputs and a host copy of the u8 output frame
  roofline  the dominant kernel class of the step against the roofline SURVEY.md 8(d) assigns to it: a6 is bounded by
            the tensor cores -- algorithmic FLOPs / CUDA-event time / sustained BF16 peak (intermediates count as zero
            bytes); `hbm_view` keeps the engineering view (bytes the kernel's dataflow must move / copy peak)
  front_c3  metric part (ii): depth-aware projection at 1080p, batch 8 (config C3's three flow fields) and the warps,
            GB/s and fractions of the measured copy peak and of the nominal 8 TB/s
  c4, c5    the other BASELINE configurations, driver-visible (N=1 only; skip with --no-extras)
  cpu_baseline  the CPU oracle on a bounded sample with all host cores (rank 0, N=1)
--dump-outputs DIR writes the u8 frames (1080x1920x3) of the last timed step, one per rank in rank order as the gather
hands them to the caller, as DIR/frames.npy in float32.  Past 64 MB (N > 2) it writes the same fixed, seeded sample of
pixels of every frame instead: DIR/frames_sample.npy (N, pixels, 3) and their flat indices, DIR/frames_sample_pixels.npy.
The inputs and weights are seeded, so two builds run with the same arguments can be compared frame for frame.
`--impl reference` times the CPU restatement (oracle/; the reference's ops on this path are CUDA-only) with all host
threads: one step = the full-size front + the conv stack (both passes) on one quarter-height band (68x480 LR pixels)
of one of the 20 maps -- a bounded sample, scaled by pixel-maps and labelled `extrapolated`.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H_LR, W_LR, T_WIN, SCALE = 270, 480, 7, 4
M_MAPS = 3 * T_WIN - 1
METRIC = "sr_frames_per_s_4x_1080p_out"
UNIT = "frames/s"
WORKLOAD = "C2: 4x VSR 480x270->1920x1080, 7-frame window (M=20 maps), batch 1 per GPU"
MAX_DISP = 8.0        # the synthetic smooth flow is scaled to max |component| = 8 px (SURVEY.md 8d)


def load_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return {"hbm": float(p["hbm_gbs"]), "bf16_burst": float(p["bf16_tflops"]),
                "bf16_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "measured"}
    except Exception:
        return {"hbm": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------------
# synthetic inputs of the C2 shape (seeded; SURVEY.md 8d)
# ------------------------------------------------------------------------------------------------
def make_inputs(seed, h=H_LR, w=W_LR, T=T_WIN):
    from video_super_resolution_b200 import synthetic as syn
    la, lb = syn.logits(h, w, seed=seed + 3)
    return {"frames": syn.frames(T, h, w, seed=seed), "flows": syn.smooth_flow(T - 1, h, w, MAX_DISP, seed=seed + 1),
            "inv_depth": syn.inv_depth(T - 1, h, w, seed=seed + 2), "logits_a": la, "logits_b": lb}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (kind "port": the reference has no CPU implementation of this path and its
# ops are CUDA-only, SURVEY.md 8c)
# ------------------------------------------------------------------------------------------------
BANDS = 4     # a CPU step covers one quarter-height band of one map (68 of 270 LR rows, full width)


class CpuFrame:
    """One C2 frame on the host, piece by piece.  step(i): the projection / warp / stack front at full size, then the
    conv stack (both passes) on ONE quarter-height band (68 x 480 LR pixels, full width) of ONE of the 20 maps.  The
    maps are independent until the per-pixel fc fuse and the stack's cost is linear in LR pixels, so a frame costs
    t_front + 20 maps x 4 bands; the bands are large enough (32 640 LR pixels, 522 240 HR pixels) for the CPU convs to
    run at their full-size efficiency -- the 24x24 crops of round 1 understated it.  A whole frame on the host is
    ~40 TFLOP of fp32 convs (minutes on 16-32 cores), so it is sampled: 80 steps would measure all of it."""

    def __init__(self, threads, seed=0):
        import torch
        from oracle import srfbn_oracle as so
        torch.set_num_threads(threads)
        self.threads = threads
        self.inp = {k: v.numpy() for k, v in make_inputs(seed).items()}
        self.sd = so.init_state_dict(num_maps=M_MAPS, seed=0)
        self.t_front, self.t_piece, self.rows = [], [], 0

    def step(self, i):
        import numpy as np
        import torch
        from oracle import oracle as orc
        from oracle import srfbn_oracle as so
        inp = self.inp
        m, band = (i // BANDS) % M_MAPS, i % BANDS
        y0, y1 = band * H_LR // BANDS, (band + 1) * H_LR // BANDS
        t0 = time.perf_counter()
        stack, _ = orc.warp_fuse_front(inp["frames"], inp["flows"], inp["inv_depth"], inp["logits_a"], inp["logits_b"], None,
                                       threads=self.threads)
        t1 = time.perf_counter()
        x = torch.from_numpy(np.ascontiguousarray(stack[m:m + 1, :, y0:y1]))
        with torch.no_grad():
            so.forward_maps(x, self.sd)         # pass 1 (video_super_resolution.py:41)
            so.forward_maps(x, self.sd)         # fuse pass (:64): same layers on the stack with the new estimate slot
        t2 = time.perf_counter()
        self.t_front.append(t1 - t0)
        self.t_piece.append(t2 - t1)
        self.rows += y1 - y0
        return t2 - t0

    def frame_seconds(self):
        """(seconds per frame, fraction of the frame's conv work measured, description)."""
        tf = sum(self.t_front) / len(self.t_front)
        tm = sum(self.t_piece)
        frac = self.rows / float(M_MAPS * H_LR)
        sec = tf + tm / frac
        desc = (f"front (projection+warp+stack) at full {W_LR}x{H_LR}: {tf:.2f} s; conv stack x2 on {len(self.t_piece)} "
                f"quarter-height bands (~{H_LR // BANDS}x{W_LR} LR pixels each, one map per band): {tm:.1f} s = "
                f"{100 * frac:.2f} % of the frame's LR pixel-maps, scaled x{1 / frac:.1f} (cost is linear in pixel-maps)")
        return sec, frac, desc


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    cpu = CpuFrame(threads)
    wall = []
    for i in range(args.warmup + args.steps):
        if i == args.warmup:
            cpu.t_front, cpu.t_piece, cpu.rows = [], [], 0          # the warm-up steps are not part of the sample
        t = cpu.step(i)
        if i >= args.warmup:
            wall.append(t)
    sec, frac, desc = cpu.frame_seconds()
    val = 1.0 / sec
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sum(wall) / len(wall) * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "step": "a bounded sample of the frame: the full front + the conv stack (both passes) on one quarter-"
                               "height band of one of the 20 maps; `value` = 1 / (front + band time scaled to 20 maps x 4 bands)",
                       "note": "CPU restatement (oracle/): the reference's ops on this path are CUDA-only"},
            "seconds_per_frame": sec, "frame_fraction_measured": frac, "extrapolated": frac < 1.0,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc,
                             "extrapolated": frac < 1.0},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler (NVML during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons during the timed region, read in-process through NVML
    (spawning nvidia-smi every 200 ms from a process that maps 20+ GB stalls the launching thread)."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._th = None
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.replace(",", "").isdigit() else index
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._max = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._h = None

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append((nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM),
                                     nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)))
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        if self._h is None:
            return
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()

    def stop(self):
        self._stop.set()
        if self._th:
            self._th.join(timeout=2)
        if self._h is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "note": "NVML unavailable"}
        nv = self._nv
        sm = sorted(s[0] for s in self.samples)
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        reasons = sorted(k for k, b in bits.items() if any(s[1] & b for s in self.samples))
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self._max, "reasons": reasons, "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# sub-records: the other BASELINE configurations, driver-visible
# ------------------------------------------------------------------------------------------------
def _median_ms(fn, iters, warm, torch):
    """ms per call: `iters` calls back to back between two CUDA events (as the bench's steps are timed), median of 3."""
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(3):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / iters)
    return sorted(ts)[1]


def front_c3(dev, peaks):
    """Metric part (ii): projection + warp GB/s against the HBM peak.  C3 = DepthProjection at 1080p, batch 8 (8 x 25 MB
    in + 8 x 35 MB out: inputs + outputs exceed the 126 MB L2), its three flow fields; the warps at the same size.
    Algorithmic bytes per pixel: SURVEY.md 8(d) (a2: 29, a3 C=3 + fused norm: 48, label warp: 10)."""
    import torch
    from video_super_resolution_b200 import ops, synthetic as syn
    B, h, w = 8, 1080, 1920
    P = B * h * w

    def rec(ms, bpp):
        gb = bpp * P / ms / 1e6
        return {"us_per_image": round(ms * 1e3 / B, 2), "GBps": round(gb, 1), "frac_hbm_measured": round(gb / peaks["hbm"], 4),
                "frac_hbm_8TBs": round(gb / 8000.0, 4)}

    out = {"config": "C3: DepthProjection (splat + normalise + hole fill) 1920x1080, batch 8, 29 B/pixel; warps at the same size",
           "hbm_peak_measured_GBps": peaks["hbm"], "timing": "20 calls back to back between two CUDA events, median of 3 repeats, after 5 warm-ups", "cases": {}}
    inv = syn.inv_depth(B, h, w, seed=9).to(dev)
    smooth = syn.smooth_flow(B, h, w, 8.0, seed=1).to(dev)
    cases = {"smooth_pm8": smooth, "iid_pm64": syn.random_flow(B, h, w, 64.0, seed=8).to(dev)}
    occ_f, occ_d = syn.occlusion_scene(B, h, w, shift=64.0, seed=5)
    for name, f in cases.items():
        out["cases"][name] = rec(_median_ms(lambda: ops.project_depth_flow(f, inv), 20, 5, torch), 29)
    occ_f, occ_d = occ_f.to(dev), occ_d.to(dev)
    out["cases"]["dense_occlusion_pm64"] = rec(_median_ms(lambda: ops.project_depth_flow(occ_f, occ_d), 20, 5, torch), 29)
    out["cases"]["smooth_pm8_tile_path(max_disp=8)"] = rec(_median_ms(lambda: ops.project_depth_flow(smooth, inv, 8.0), 20, 5, torch), 29)
    src = (torch.rand((B, h, w, 3), device=dev) * 255)
    out["cases"]["warp_C3_fast+resid_norm"] = rec(_median_ms(lambda: ops.warp(src, smooth, 2, ref=src), 20, 5, torch), 48)
    lab = syn.labels(B, h, w).to(dev)
    out["cases"]["label_warp_u8"] = rec(_median_ms(lambda: ops.warp_labels(lab, smooth), 20, 5, torch), 10)
    return out


def sub_c4(dev, peaks, steps=2):
    """C4: 2x VSR 1920x1080 -> 3840x2160, 5-frame window (M = 14), one window on this GPU."""
    import gc
    import torch
    from video_super_resolution_b200 import synthetic as syn
    from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
    from video_super_resolution_b200.pipeline import WarpFusePipeline
    T, h, w, s = 5, 1080, 1920, 2
    M = 3 * T - 1
    torch.manual_seed(0)
    sr = _gained(SRProjectionModule(num_maps=M, upscale_factor=s))
    pipe = WarpFusePipeline(T, h, w, sr, s, device=dev, max_disp=MAX_DISP)
    la, lb = syn.logits(h, w, seed=3)
    inp = [syn.frames(T, h, w, seed=0).to(dev), syn.smooth_flow(T - 1, h, w, MAX_DISP, seed=1).to(dev),
           syn.inv_depth(T - 1, h, w, seed=2).to(dev), la.to(dev), lb.to(dev)]
    pipe.step(*inp)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        pipe.step(*inp)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    flops = 2 * M * h * w * 3.575e6     # SURVEY.md 8 a6: 3.575 MFLOP per LR pixel per map at x2, two passes
    rec = {"config": "C4: 2x VSR 1920x1080->3840x2160, 5-frame window (M=14), one window per GPU (SRFBN k6 s2 p2)",
           "metric": "sr_frames_per_s_2x_4k_out", "value": 1e3 / ms, "unit": UNIT, "ms_per_step": ms, "steps": steps,
           "tflops_per_step": flops / 1e12, "step_tensor_frac": flops / ms / 1e9 / peaks["bf16_sustained"]}
    del pipe, sr, inp
    gc.collect()
    torch.cuda.empty_cache()
    return rec


def sub_c5(dev, rank, world, frames=300):
    """C5: 300-frame 720x360 -> 2880x1440 4x sequence, T = 3 windows (M = 8), the reference's 20 chunks with the
    recurrence reset at chunk starts (main.py:196), sharded over the ranks (strong scaling); pinned-host inputs and
    the NCCL gather of the u8 frames inside the timed region."""
    import torch
    import torch.distributed as dist
    from video_super_resolution_b200 import synthetic as syn
    from video_super_resolution_b200.network.video_super_resolution import VSR
    from video_super_resolution_b200.pipeline import gather_frames_ragged, run_sequence, shard_chunks_even
    from video_super_resolution_b200.utils.video_utils import chunk_windows
    T, h, w, s, n = 3, 360, 720, 4, frames
    torch.manual_seed(0)
    vsr = VSR(window=T)
    _gained(vsr.model)
    chunks = chunk_windows(n, T)
    mine = shard_chunks_even(chunks, world, rank)
    lo = min(c.start for c in mine)
    hi = max(c.stop for c in mine) + T - 1                # frames this rank needs (T-1 halo frames, replicated)
    g = torch.Generator().manual_seed(7)
    frames_u8 = torch.randint(0, 256, (n, h, w, 3), generator=g, dtype=torch.uint8).pin_memory()
    flows_h = syn.smooth_flow(n - 1, h, w, MAX_DISP, seed=1).pin_memory()
    inv_h = syn.inv_depth(n - 1, h, w, seed=2).pin_memory()
    la, lb = (t.to(dev) for t in syn.logits(h, w, seed=3))
    local = [range(c.start - lo, c.stop - lo) for c in mine]
    out = torch.empty((sum(len(c) for c in mine), s * h, s * w, 3), dtype=torch.uint8, device=dev)
    vsr._pipe(h, w, dev).max_disp = MAX_DISP

    def one_pass():
        fr = frames_u8[lo:hi].to(dev, non_blocking=True).to(torch.float32)
        fl = flows_h[lo:hi - 1].to(dev, non_blocking=True)
        iv = inv_h[lo:hi - 1].to(dev, non_blocking=True)
        run_sequence(vsr, fr, fl, iv, lambda k: (la, lb), local, out=out)
        return gather_frames_ragged(out)

    fr = frames_u8[lo:lo + T + 2].to(dev).to(torch.float32)      # warm-up: three windows
    run_sequence(vsr, fr, flows_h[lo:lo + T + 1].to(dev), inv_h[lo:lo + T + 1].to(dev), lambda k: (la, lb), [range(0, 3)])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    allf = one_pass()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    n_out = n - T + 1
    assert allf.shape[0] == n_out
    return {"config": f"C5: {n}-frame 720x360 -> 2880x1440 4x sequence, 3-frame windows (M=8), reference chunking (20 chunks, "
                      "recurrence reset at chunk starts), even shards; host (pinned) u8 frames + geometry in, u8 frame "
                      "all-gather inside the timed region", "metric": "sr_frames_per_s_4x_sequence", "unit": UNIT,
            "n_gpus": world, "value": n_out / (ms / 1e3), "seconds_per_sequence": ms / 1e3, "scaling": "strong",
            "gathered_bytes": int(allf.numel())}


DUMP_LIMIT_BYTES = 64 << 20


def dump_frames(out_dir, frames):
    """frames (N,H,W,C) u8 -> out_dir/frames.npy in float32, or, past DUMP_LIMIT_BYTES, the same fixed, seeded sample
    of pixels of every frame (frames_sample.npy, (N,pixels,C)) with their flat indices (frames_sample_pixels.npy)."""
    import numpy as np
    import torch
    n, h, w, c = frames.shape
    os.makedirs(out_dir, exist_ok=True)
    if frames.numel() * 4 <= DUMP_LIMIT_BYTES:
        np.save(os.path.join(out_dir, "frames.npy"), frames.float().cpu().numpy())
        return
    k = DUMP_LIMIT_BYTES // (n * c * 4 + 8)                   # float32 values of every frame + one float64 index
    pix = np.sort(np.random.default_rng(0).choice(h * w, size=k, replace=False))
    sample = frames.reshape(n, h * w, c)[:, torch.from_numpy(pix).to(frames.device)]
    np.save(os.path.join(out_dir, "frames_sample.npy"), sample.float().cpu().numpy())
    np.save(os.path.join(out_dir, "frames_sample_pixels.npy"), pix.astype(np.float64))


def _gained(sr, gain=2.3):
    """x2.3 so that a 40-layer random net keeps O(1) activations (the reference's default initialisers decay)."""
    import torch
    with torch.no_grad():
        for name, p in sr.named_parameters():
            if name.endswith(".0.weight") and not name.startswith(("sub_mean", "add_mean")):
                p.mul_(gain)
    return sr


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from video_super_resolution_b200 import _lib
    from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
    from video_super_resolution_b200.pipeline import WarpFusePipeline, gather_frames

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries the one JSON line: NCCL's banner / debug output goes to stderr.  A caller-set NCCL_DEBUG is
        # kept (the driver reads the communicator's rank count from the INFO lines).
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        # NCCL prints its version banner with printf to fd 1 when the first communicator comes up: point fd 1 at
        # stderr until the warm-up collective has run, then give stdout back to the JSON line
        sys.stdout.flush()
        saved_stdout_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()

    torch.manual_seed(0)
    sr = _gained(SRProjectionModule(num_maps=M_MAPS))          # the reference's default initialisers
    pipe = WarpFusePipeline(T_WIN, H_LR, W_LR, sr, SCALE, device=dev, max_disp=MAX_DISP)
    HW3 = (SCALE * H_LR, SCALE * W_LR, 3)

    # three seeded input sets, rotated step by step (SURVEY.md 8d: seeds 0,1,2)
    SEEDS = 3
    host = [{k: v.pin_memory() for k, v in make_inputs(seed=100 * (s + 1) + rank).items()} for s in range(SEEDS)]
    res = [{k: v.to(dev) for k, v in hs.items()} for hs in host]
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())
    frames_u8 = torch.empty((args.steps,) + HW3, dtype=torch.uint8, device=dev)   # this rank's output frames
    d2h = frames_u8[0].numel()
    counters = {"k": 0}

    def step_resident():
        k = counters["k"]
        counters["k"] = k + 1
        r = res[k % SEEDS]
        counters["last"] = pipe.step(r["frames"], r["flows"], r["inv_depth"], r["logits_a"], r["logits_b"],
                                     out_u8=frames_u8[k % frames_u8.shape[0]], want_f32=False)
        return counters["last"]

    # End-to-end loop: every step's inputs come from pinned host memory and every step's u8 frame goes back to the
    # host, inside the timed region -- double-buffered on a copy stream, so that the H2D of step k+1 and the D2H of
    # step k run under the kernels of their neighbours (what a streaming caller does; utils/video_utils.py
    # PinnedFrameRing is the same scheme).  The timed region ends after the last D2H has completed.
    stage2 = [{k: torch.empty_like(v, device=dev) for k, v in host[0].items()} for _ in range(2)]
    out_host2 = [torch.empty(HW3, dtype=torch.uint8).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    e2e_state = {"k": 0, "in_ready": [None, None], "done": [None, None]}

    def e2e_prefetch(slot, k):
        with torch.cuda.stream(copy_stream):
            if e2e_state["done"][slot] is not None:
                copy_stream.wait_event(e2e_state["done"][slot])      # the step that read this slot has finished
            hs = host[k % SEEDS]
            for name in hs:
                stage2[slot][name].copy_(hs[name], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        e2e_state["in_ready"][slot] = ev

    def step_e2e():
        st = e2e_state
        k = st["k"]
        slot = k & 1
        if st["in_ready"][slot] is None:                              # first step of a run: nothing was prefetched
            e2e_prefetch(slot, k)
        cur = torch.cuda.current_stream(dev)
        cur.wait_event(st["in_ready"][slot])
        st["in_ready"][slot] = None
        sg = stage2[slot]
        y = pipe.step(sg["frames"], sg["flows"], sg["inv_depth"], sg["logits_a"], sg["logits_b"],
                      out_u8=frames_u8[k % frames_u8.shape[0]], want_f32=False)
        done = torch.cuda.Event()
        done.record(cur)
        st["done"][slot] = done
        e2e_prefetch(slot ^ 1, k + 1)                                 # next step's inputs, under this step's kernels
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(done)
            out_host2[slot].copy_(y, non_blocking=True)               # this step's frame, under the next step's kernels
        st["k"] = k + 1
        return y

    def e2e_drain():
        torch.cuda.current_stream(dev).wait_stream(copy_stream)       # the timed region includes the last D2H
        e2e_state["in_ready"] = [None, None]
        e2e_state["k"] = 0

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        counters["k"] = 0
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if world > 1:
            gather_frames(frames_u8[:steps])
        if fn is step_e2e:
            e2e_drain()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # warm-up (also builds the plan, packs weights, sets kernel attributes)
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_resident()
    if world > 1:                                 # the first collective builds NCCL's channels: not part of a step
        gather_frames(frames_u8[:1])
        torch.cuda.synchronize()
        sys.stdout.flush()
        os.dup2(saved_stdout_fd, 1)
        os.close(saved_stdout_fd)
    step_e2e()
    e2e_drain()
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    _lib.launch_count_reset()
    ms_total = timed(step_resident, args.steps)
    launches = _lib.launch_count()
    if args.dump_outputs:
        # every rank's frame of the last timed step, gathered before the e2e loop reuses its buffer
        last = gather_frames(counters["last"].unsqueeze(0))
        if rank == 0:
            dump_frames(args.dump_outputs, last)
    ms_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else None

    # the same step with the fuse pass reusing what pass 1 already convolved (pipeline.WarpFusePipeline reuse=...): NOT
    # the headline -- `value` recomputes every map in both passes, as the reference's two SRProjectionModule calls do
    reuse = None
    if not args.no_extras:
        reuse = {"note": "same C2 step, inputs resident; the M maps are independent until the per-pixel fc, so maps that enter "
                         "both passes unchanged are convolved once (bit-identical frames, tests/test_pipeline_gpu.py). "
                         "'frames': the T frame maps (video_super_resolution.py:62 feeds `data` unchanged); 'unchanged': all "
                         "but the estimate slot (this pipeline's flow / depth maps are inputs, not re-estimated). "
                         "maps_convolved_per_frame counts both passes (headline: 2 M)."}
        n_re = args.steps
        for mode, n_maps in (("frames", 2 * M_MAPS - T_WIN), ("unchanged", M_MAPS + 1)):
            pipe_r = WarpFusePipeline(T_WIN, H_LR, W_LR, sr, SCALE, device=dev, max_disp=MAX_DISP, reuse=mode)

            def step_reuse():
                k = counters["k"]
                counters["k"] = k + 1
                r = res[k % SEEDS]
                return pipe_r.step(r["frames"], r["flows"], r["inv_depth"], r["logits_a"], r["logits_b"],
                                   out_u8=frames_u8[k % frames_u8.shape[0]], want_f32=False)
            for _ in range(3):
                step_reuse()
            ms_r = timed(step_reuse, n_re)
            reuse[mode] = {"value": world * n_re / (ms_r / 1e3), "unit": UNIT, "ms_per_step": ms_r / n_re, "steps": n_re,
                           "maps_convolved_per_frame": n_maps}
            del pipe_r

    # per-launch accounting of one more step (events recorded by the library on the launching stream)
    sr.profile(True)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    r0 = res[0]
    evs[0].record()
    pipe.project_and_warp(r0["frames"], r0["flows"], r0["inv_depth"], r0["logits_a"], r0["logits_b"])
    evs[1].record()
    prof_ms = {}
    for _ in range(2):                      # the two passes of the step
        sr(pipe.stack)
        for k, d in sr.profile_read().items():
            a = prof_ms.setdefault(k, {"ms": 0.0, "launches": 0, "flops": 0.0, "bytes": 0.0})
            for f in a:
                a[f] += d[f]
    torch.cuda.synchronize()
    sr.profile(False)
    front_ms = evs[0].elapsed_time(evs[1])

    extras = {}
    if not args.no_extras:
        del pipe, stage2, res
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        if world == 1:
            extras["front_c3"] = front_c3(dev, peaks)
            torch.cuda.empty_cache()
            extras["c4"] = sub_c4(dev, peaks)
        extras["c5"] = sub_c5(dev, rank, world)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    P = H_LR * W_LR
    front_bytes = (T_WIN - 1) * P * (21 + 29 + 48) + P * 10 + P * 8 + M_MAPS * 3 * P * 4
    kernels = {"front(projection+chain+warp+mask+stack)": {"ms": front_ms, "GBps": front_bytes / front_ms / 1e6,
                                                           "frac_hbm": front_bytes / front_ms / 1e6 / peaks["hbm"],
                                                           "note": "launch-latency bound at the C2 size; see front_c3"}}
    dom, dom_ms = None, -1.0
    for k, d in prof_ms.items():
        if d["launches"] == 0 or d["ms"] <= 0:
            continue
        tf = d["flops"] / d["ms"] / 1e9
        gb = d["bytes"] / d["ms"] / 1e6
        kernels[k] = {"ms": round(d["ms"], 3), "launches": d["launches"], "TFLOPs": round(tf, 1), "GBps": round(gb, 1),
                      "frac_tensor": round(tf / peaks["bf16_sustained"], 4), "frac_hbm": round(gb / peaks["hbm"], 4)}
        if d["ms"] > dom_ms:
            dom, dom_ms = k, d["ms"]
    d = prof_ms[dom]
    # SURVEY.md 8(d): a6 (every kernel class of the conv stack) is bounded by the tensor cores; its algorithmic work is
    # the layer's 2*MAC FLOPs, intermediates count as zero bytes.  peak = sustained BF16 (the kernel is timed inside a
    # long step under the power cap).
    ach = d["flops"] / d["ms"] / 1e9
    gbs = d["bytes"] / d["ms"] / 1e6
    roof = {"bound": "tensor", "achieved": ach, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
            "frac": ach / peaks["bf16_sustained"], "traffic": None,
            "hbm_view": {"achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"],
                         "note": "bytes this kernel's dataflow must move (its HR feature-map inputs are intermediates of the "
                                 "stack, which SURVEY.md 8(d) counts as zero) / measured copy peak: the engineering view"}}
    # DRAM bytes per launch of that kernel class from the committed ncu capture of the same shapes
    # (dram__bytes_read.sum + dram__bytes_write.sum, one pass, C2 size; tools/traffic_json.py)
    try:
        pat = {"fused_downtran_conv8x8s4": "fused_down_kernel", "deconv8x8s4": "igemm_kernel<1, 32, 256>",
               "pointwise_lr": "igemm_kernel<0, 32, 32>", "finalize_lr": "finalize_lr_kernel",
               "conv_out3x3": "igemm_kernel<2, 32, 32>", "conv_in_gemm": "igemm_kernel<0, 32, 128>",
               "fc_fuse": "fc_fuse_kernel", "im2col": "im2col_kernel"}[dom]
        tfile = next(f for f in ("traffic_r02h.json", "traffic_r02.json", "traffic_r01h.json", "traffic_r01f.json")
                     if os.path.exists(os.path.join(ROOT, "profiles", f)))
        tr = [t["dram_read_bytes"] + t["dram_write_bytes"]
              for t in json.load(open(os.path.join(ROOT, "profiles", tfile))) if pat in t["kernel"]]
        roof["traffic"] = sum(tr) / len(tr) if tr else None
        roof["traffic_source"] = f"profiles/{tfile} (ncu, same shapes, average over the class's launches)"
    except Exception:
        pass
    roof.update({"kernel": dom, "launches_per_step": d["launches"], "avg_launch_ms": d["ms"] / d["launches"],
                 "algorithmic_per_launch": {"flops": d["flops"] / d["launches"], "bytes": d["bytes"] / d["launches"]},
                 "peak_source": peaks["source"] + " (MEASURED_PEAKS.json: sustained bf16 / copy GB/s)",
                 "share_of_step": d["ms"] / (ms_total / args.steps)})

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        c = CpuFrame(threads)
        for i in range(3):                        # three quarter-map bands, all cores: ~10-20 s
            c.step(i)
        sec, frac, desc = c.frame_seconds()
        cpu = {"value": 1.0 / sec, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc, "extrapolated": True}

    flops_step = sum(v["flops"] for v in prof_ms.values())
    line = {"metric": METRIC, "value": world * args.steps / (ms_total / 1e3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "l2": "working set (~22 GB of activations per step) exceeds the 126 MB L2; no flush needed",
                       "inputs": "3 seeded input sets rotated step by step",
                       "weights": "random init (reference initialisers x2.3 gain), BF16 operands / FP32 accumulate",
                       "steps_per_frame": "projection+warp front, conv stack x2 (pass 1 + fuse pass), 3 feedback steps"},
            "e2e": {"value": world * args.steps / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "kernels": kernels, "tflops_per_step": flops_step / 1e12,
            "step_tensor_frac": flops_step / (ms_total / args.steps) / 1e9 / peaks["bf16_sustained"]}
    if reuse is not None:
        line["c2_reuse"] = reuse
    line.update(extras)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the front_c3 / c4 / c5 sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write every rank's output frame of the last timed step to DIR/frames.npy (float32, values "
                         "0..255; a seeded pixel sample past 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the frames of the b200 arm; the reference arm computes a sample of a frame")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
