"""Device timing of the deterministic projection and Resample2d input gradient against the default paths (CUDA events).
Writes one JSON line (default profiles/time_deterministic.json) with the card's name and power limit read in the same
run; the human-readable lines go to stdout.

    python tools/time_deterministic.py [--out PATH]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from video_super_resolution_b200 import ops, synthetic as syn  # noqa: E402
from tools.time_ops import timeit  # noqa: E402

DEV = "cuda:0"


def card():
    """Name, power limit and max SM clock of cuda:0 (read only)."""
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    fields = [f.strip() for f in r.stdout.strip().split(",")] if r.returncode == 0 else []
    return {"name": torch.cuda.get_device_name(0), "power_limit": fields[1] if len(fields) > 1 else "unknown",
            "max_sm_clock": fields[2] if len(fields) > 2 else "unknown"}


def projection(res):
    B, h, w = 8, 1080, 1920
    fields = {"smooth8": syn.smooth_flow(B, h, w, 8.0, seed=0), "iid64": syn.random_flow(B, h, w, 64.0, seed=1),
              "occlusion64": syn.occlusion_scene(B, h, w, 64.0, seed=2)[0]}
    inv = syn.inv_depth(B, h, w, seed=3).to(DEV)
    for name, f in fields.items():
        f = f.to(DEV)
        for weighted in (False, True):
            d = inv if weighted else None
            paths = {"general": lambda: ops.project_flow(f, d, None, deterministic=False),
                     "tile(max_disp=8)": lambda: ops.project_flow(f, d, 8.0, deterministic=False),
                     "deterministic": lambda: ops.project_flow(f, d, deterministic=True)}
            for p, fn in paths.items():
                us = timeit(fn) * 1e3 / B
                key = f"projection_1080p_B8_{name}_{'depth' if weighted else 'flow'}_{p}_us_per_image"
                res[key] = round(us, 1)
                print(f"{key:75s} {us:10.1f}", flush=True)


def resample(res):
    g = torch.Generator().manual_seed(5)
    B, C, H, W = 1, 3, 1080, 1920
    x = (torch.rand((B, C, H, W), generator=g) * 255).to(DEV)
    flow = ((torch.rand((B, 2, H, W), generator=g) * 2 - 1) * 64).to(DEV)
    go = torch.randn((B, C, H, W), generator=g).to(DEV)
    for p, det in (("atomic", False), ("deterministic", True)):
        ms = timeit(lambda: ops.resample2d_backward(x, flow, go, deterministic=det))
        key = f"resample2d_backward_1080p_C3_iid64_{p}_ms"
        res[key] = round(ms, 3)
        print(f"{key:75s} {ms:10.3f}", flush=True)


def skew(res):
    # projection: every source of the image lands in one cell
    for n in (256, 1080):
        h, w = n, n * 16 // 9 if n == 1080 else n
        ys, xs = torch.meshgrid(torch.arange(h, dtype=torch.float32), torch.arange(w, dtype=torch.float32), indexing="ij")
        f = torch.stack((100.5 - xs, 60.25 - ys), dim=-1)[None].contiguous().to(DEV)
        ms = timeit(lambda: ops.project_flow(f, deterministic=True), iters=5, warm=1)
        key = f"projection_skew_one_cell_{h}x{w}_deterministic_ms"
        res[key] = round(ms, 3)
        print(f"{key:75s} {ms:10.3f}", flush=True)
    # resample gradient: every sample outside the image -> one border pixel receives them all
    for H, W in ((256, 256), (1080, 1920)):
        g = torch.Generator().manual_seed(6)
        x = torch.rand((1, 3, H, W), generator=g).to(DEV)
        go = torch.randn((1, 3, H, W), generator=g).to(DEV)
        flow = torch.full((1, 2, H, W), 1.0e4, device=DEV)
        for p, det in (("atomic", False), ("deterministic", True)):
            ms = timeit(lambda: ops.resample2d_backward(x, flow, go, deterministic=det), iters=5, warm=1)
            key = f"resample2d_backward_skew_all_outside_{H}x{W}_C3_{p}_ms"
            res[key] = round(ms, 3)
            print(f"{key:75s} {ms:10.3f}", flush=True)


def c2_step(res):
    from oracle import srfbn_oracle as so
    from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
    from video_super_resolution_b200.pipeline import WarpFusePipeline
    T, h, w = 7, 270, 480
    M = 3 * T - 1
    sr = SRProjectionModule(num_maps=M)
    sr.load_state_dict(so.init_state_dict(num_maps=M, seed=0, gain=2.3))
    la, lb = syn.logits(h, w, seed=4)
    fields = {"smooth8": syn.smooth_flow(T - 1, h, w, 8.0, seed=2), "iid64": syn.random_flow(T - 1, h, w, 64.0, seed=2)}
    fr, inv = syn.frames(T, h, w, seed=1).to(DEV), syn.inv_depth(T - 1, h, w, seed=3).to(DEV)
    u8 = torch.empty((4 * h, 4 * w, 3), dtype=torch.uint8, device=DEV)
    for name, fl in fields.items():
        args = (fr, fl.to(DEV), inv, la.to(DEV), lb.to(DEV))
        for max_disp in (None, 8.0) if name == "smooth8" else (None,):
            pipe = WarpFusePipeline(T, h, w, sr, 4, device=DEV, max_disp=max_disp)
            for flag in (False, True):
                torch.use_deterministic_algorithms(flag)
                try:
                    ms = timeit(lambda: pipe.step(*args, out_u8=u8, want_f32=False), iters=10, warm=3)
                finally:
                    torch.use_deterministic_algorithms(False)
                key = f"c2_step_{name}_max_disp_{max_disp}_flag_{'on' if flag else 'off'}_frames_per_s"
                res[key] = round(1e3 / ms, 2)
                print(f"{key:75s} {1e3 / ms:10.2f}", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "time_deterministic.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    res = {"tool": "tools/time_deterministic.py", "date": time.strftime("%Y-%m-%d"), "card": card(),
           "timing": "CUDA events, median of 20 calls after 5 warm-up calls (skew: 5 after 1; C2 step: 10 after 3)"}
    print(json.dumps(res["card"]), flush=True)
    projection(res)
    resample(res)
    skew(res)
    c2_step(res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
