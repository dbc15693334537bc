#!/usr/bin/env python
"""Throughput of the window-batched step: W frame windows per WarpFusePipeline step, eager and as a GraphedStep.

    python tools/bench_windows.py [--windows 1 2 4 8] [--configs c1 s320 c2 c5] [--min-ms 1000] [--out FILE]

Configurations (x4, synthetic seeded inputs, smooth +-8 px flows, max_disp = 8):
    c1    LR 64x64,   T = 3  (BASELINE C1's frame size)
    s320  LR 320x180, T = 3  (-> 1280x720)
    c2    LR 480x270, T = 7  (BASELINE C2)
    c5    LR 720x360, T = 3  (BASELINE C5's frames)
One JSON line per (config, W, mode) on stdout (and appended to --out): ms per step and frames/s (W frames per step),
device time from CUDA events over at least --min-ms of steps after a warm-up; the library's kernel launches per eager
step (vsr_launch_count; a graph replay is one graph launch); the card's name and power limit, read in the same run.
The conv-stack workspace is capped (--cap-gb) so that large W fit: the plan then sweeps its maps in chunks (the
`chunk_maps` field).  Inputs are the same every step; at c1 the working set stays in the 126 MB L2."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {"c1": (64, 64, 3), "s320": (180, 320, 3), "c2": (270, 480, 7), "c5": (360, 720, 3)}
MAX_DISP = 8.0


def card():
    import torch
    name, limit = torch.cuda.get_device_name(0), None
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        if r.returncode == 0 and r.stdout.strip():
            name, limit = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
    except (OSError, subprocess.TimeoutExpired):
        pass
    return name, limit


def gained(sr, gain=2.3):
    import torch
    with torch.no_grad():
        for n, p in sr.named_parameters():
            if n.endswith(".0.weight") and not n.startswith(("sub_mean", "add_mean")):
                p.mul_(gain)
    return sr


def timed(fn, min_ms, torch):
    """ms per call: a short probe sizes a timed window of at least min_ms."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        fn()
    e1.record()
    torch.cuda.synchronize()
    n = max(5, min(2000, int(min_ms / max(e0.elapsed_time(e1) / 3, 1e-3)) + 1))
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, n


def run(cfg, W, args, name, limit, out):
    import torch
    from video_super_resolution_b200 import _lib, synthetic as syn
    from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
    from video_super_resolution_b200.pipeline import GraphedStep, WarpFusePipeline
    h, w, T = CONFIGS[cfg]
    dev = torch.device("cuda:0")
    M, s = 3 * T - 1, 4
    sr = gained(SRProjectionModule(num_maps=M, workspace_cap_bytes=int(args.cap_gb * (1 << 30))))
    pipe = WarpFusePipeline(T, h, w, sr, s, device=dev, max_disp=MAX_DISP, windows=W)
    wins = []
    for b in range(W):
        la, lb = syn.logits(h, w, seed=10 * b + 4)
        wins.append([syn.frames(T, h, w, seed=10 * b), syn.smooth_flow(T - 1, h, w, MAX_DISP, seed=10 * b + 1),
                     syn.inv_depth(T - 1, h, w, seed=10 * b + 2), la, lb])
    inp = [torch.stack(list(p)).to(dev).contiguous() for p in zip(*wins)]
    if W == 1:
        inp = [t[0] for t in inp]
    u8 = torch.empty(((W,) if W > 1 else ()) + (s * h, s * w, 3), dtype=torch.uint8, device=dev)

    def step():
        pipe.step(*inp, out_u8=u8, want_f32=False)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    _lib.launch_count_reset()
    step()
    torch.cuda.synchronize()
    launches = _lib.launch_count()
    ent = next(iter(sr._plans.values()))
    base = {"config": cfg, "lr": [h, w], "T": T, "scale": s, "windows": W, "card": name, "power_limit": limit,
            "launches_per_step": launches, "chunk_maps": ent["chunk_maps"], "maps": W * M}
    ms, n = timed(step, args.min_ms, torch)
    lines = [dict(base, mode="eager", ms_per_step=round(ms, 4), frames_per_s=round(W * 1000.0 / ms, 2), steps=n)]
    g = GraphedStep(pipe, want_f32=False, warmup=args.warmup)
    g.load(*inp)
    ms, n = timed(g.replay, args.min_ms, torch)
    lines.append(dict(base, mode="graph", ms_per_step=round(ms, 4), frames_per_s=round(W * 1000.0 / ms, 2), steps=n))
    for ln in lines:
        s_ = json.dumps(ln)
        print(s_, flush=True)
        if out:
            out.write(s_ + "\n")
            out.flush()
    del g, pipe, sr, inp, u8
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--windows", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--configs", nargs="+", default=list(CONFIGS), choices=list(CONFIGS))
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--min-ms", type=float, default=1000.0)
    ap.add_argument("--cap-gb", type=float, default=40.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_windows.py measures on the GPU; no CUDA device here")
    name, limit = card()
    out = open(args.out, "a") if args.out else None
    with torch.no_grad():
        for cfg in args.configs:
            for W in args.windows:
                run(cfg, W, args, name, limit, out)
    if out:
        out.close()


if __name__ == "__main__":
    main()
