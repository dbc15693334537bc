#!/usr/bin/env python
"""Throughput of ONE recurrence (a chunk: window k+1 takes window k's output as its estimate) run map-parallel over a
map group of G GPUs (DESIGN.md 11).

    python -m torch.distributed.run --nproc_per_node G tools/bench_map_parallel.py [--configs c2 c5] [--out FILE]
    python tools/bench_map_parallel.py --rank0-compute 2 4 8 [--configs c2 c5] [--out FILE]

Configurations (x4, synthetic seeded inputs, smooth +-8 px flows, max_disp = 8, as tools/bench_windows.py):
    c2    LR 480x270, T = 7, M = 20 maps  (BASELINE C2)
    c5    LR 720x360, T = 3, M = 8 maps   (BASELINE C5's frames)
Under torch.distributed.run (G = world size, one GPU per rank): one JSON line per (config, reuse) with ms per frame and
frames/s of the recurrence, and the per-step split from CUDA events on rank 0's stream, each stage summed over the
timed steps and divided by their number: `front` (a1-a5 + a7 on rank 0), `broadcast` (stack + mask), `sweep` (the conv
stack over the rank's maps, both passes; the slowest rank's), `exchange` (the all_to_all of both passes), `gathers`
(estimate slots and the u8 frame), `other` (pack, band fuse, slot and reorder kernels).  A collective's time includes
waiting for the slowest peer.  Without torch.distributed.run the one-GPU recurrence (no group) is measured as the
baseline.  --rank0-compute G...: on one GPU, rank 0's share of the work of a group of G (its ceil(M/G) maps, its band,
the front) with the collectives left out -- the compute bound of the scaling, not a multi-GPU measurement.
The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_windows import MAX_DISP, card, gained  # noqa: E402

CONFIGS = {"c2": (270, 480, 7), "c5": (360, 720, 3)}
STAGES = ("front", "broadcast", "sweep", "exchange", "gathers")


class _Timed:
    """Wraps a MapGroup (or a stand-in) and records CUDA events around each collective, by stage."""

    def __init__(self, g, ev):
        self.g, self.ev, self.rank, self.size = g, ev, g.rank, g.size

    def _t(self, stage, fn, *a):
        import torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(*a)
        e1.record()
        self.ev.append((stage, e0, e1))

    def broadcast(self, t, src=0):
        self._t("broadcast", self.g.broadcast, t, src)

    def all_to_all(self, out, inp, out_splits, in_splits):
        self._t("exchange", self.g.all_to_all, out, inp, out_splits, in_splits)

    def all_gather(self, out, inp):
        self._t("gathers", self.g.all_gather, out, inp)


class _NoComm:
    """Rank 0 of a group of `size` whose collectives move nothing (--rank0-compute)."""

    def __init__(self, size):
        self.rank, self.size = 0, size

    def broadcast(self, t, src=0):
        pass

    def all_to_all(self, out, inp, out_splits, in_splits):
        pass

    def all_gather(self, out, inp):
        pass


def _wrap(obj, name, stage, ev):
    import torch
    fn = getattr(obj, name)

    def timed(*a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn(*a, **k)
        e1.record()
        ev.append((stage, e0, e1))
        return r
    setattr(obj, name, timed)


def run(cfg, reuse, G, mg, args, name, limit, out, mode):
    import torch
    import torch.distributed as dist
    from video_super_resolution_b200 import synthetic as syn
    from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
    from video_super_resolution_b200.pipeline import WarpFusePipeline
    h, w, T = CONFIGS[cfg]
    dev = torch.device("cuda", torch.cuda.current_device())
    M, s = 3 * T - 1, 4
    ev = []
    tg = _Timed(mg, ev) if mg is not None else None
    torch.manual_seed(0)
    sr = gained(SRProjectionModule(num_maps=M, map_group=tg))
    pipe = WarpFusePipeline(T, h, w, sr, s, device=dev, max_disp=MAX_DISP, reuse=reuse, map_group=tg)
    _wrap(pipe, "project_and_warp", "front", ev)
    _wrap(sr, "_sweep", "sweep", ev)
    la, lb = syn.logits(h, w, seed=4)
    inp = [t.to(dev).contiguous() for t in (syn.frames(T, h, w, seed=0), syn.smooth_flow(T - 1, h, w, MAX_DISP, seed=1),
                                            syn.inv_depth(T - 1, h, w, seed=2), la, lb)]
    u8 = torch.empty((s * h, s * w, 3), dtype=torch.uint8, device=dev)
    state = {"est": None}

    def step():                       # one window of the recurrence: the previous output is the estimate
        if tg is None:
            y = pipe.step(*inp, estimate_hr=None if state["est"] is None else state["est"][0], out_u8=u8)
        else:
            y = pipe.step(*inp, estimate_hr_band=state["est"], out_u8=u8, gather="u8")
        state["est"] = y

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if mg is not None and mode == "nccl":
        dist.barrier()
    ev.clear()
    n = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    split = {k: 0.0 for k in STAGES}
    for stage, a, b in ev:
        split[stage] += a.elapsed_time(b) / n
    if mode == "nccl" and G > 1:
        t = torch.tensor([split["sweep"]], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)   # the slowest rank's sweep
        split["sweep"] = float(t)
    split["other"] = ms - sum(split.values())
    if mg is not None and mode == "nccl" and mg.rank != 0:
        return
    ln = {"config": cfg, "lr": [h, w], "T": T, "maps": M, "scale": s, "G": G, "reuse": reuse, "mode": mode,
          "maps_per_rank": -(-M // G), "ms_per_frame": round(ms, 3), "frames_per_s": round(1000.0 / ms, 2),
          "steps": n, "split_ms": {k: round(v, 3) for k, v in split.items()}, "card": name, "power_limit": limit}
    line = json.dumps(ln)
    print(line, flush=True)
    if out:
        out.write(line + "\n")
        out.flush()
    del pipe, sr, inp, u8, state
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--configs", nargs="+", default=list(CONFIGS), choices=list(CONFIGS))
    ap.add_argument("--reuse", nargs="+", default=["none", "frames"], choices=["none", "frames"])
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rank0-compute", type=int, nargs="*", default=None, metavar="G")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_map_parallel.py measures on the GPU; no CUDA device here")
    distributed = "WORLD_SIZE" in os.environ
    if distributed:
        import torch.distributed as dist
        from video_super_resolution_b200.map_parallel import MapGroup
        rank = int(os.environ["RANK"])
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    name, limit = card()
    out = open(args.out, "a") if args.out and (not distributed or int(os.environ["RANK"]) == 0) else None
    t0 = time.time()
    try:
        with torch.no_grad():
            for cfg in args.configs:
                for reuse in args.reuse:
                    r = None if reuse == "none" else reuse
                    if distributed:
                        mg = MapGroup(dist.group.WORLD)
                        run(cfg, r, mg.size, mg, args, name, limit, out, "nccl")
                    elif args.rank0_compute:
                        for G in args.rank0_compute:
                            run(cfg, r, G, _NoComm(G), args, name, limit, out, "rank0_compute_only")
                    else:
                        run(cfg, r, 1, None, args, name, limit, out, "one_gpu")
    finally:
        if out:
            out.close()
        if distributed:
            dist.destroy_process_group()
    print(f"# {time.time() - t0:.1f} s", file=sys.stderr)


if __name__ == "__main__":
    main()
