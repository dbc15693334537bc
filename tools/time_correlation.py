"""Device time of the FlowNetC cost volume (256 x 135 x 240, pad 20, max displacement 20, strides 1/2): the
register-tiled kernel, the generic kernel (VSR_CORR_GENERIC=1), the backward (both input gradients) and the reference
binary (oracle/_ref) when present.  Prints the GPU's name and power limit first: the times belong to them."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from video_super_resolution_b200 import ops  # noqa: E402


def timed(fn, n=50):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    props = torch.cuda.get_device_properties(0)
    try:
        import subprocess
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip()
    except OSError:  # pragma: no cover
        power = "unknown"
    print(f"{props.name}, power limit {power or 'unknown'}")
    B, C, H, W = 1, 256, 135, 240
    a, b = torch.randn((B, C, H, W), device="cuda"), torch.randn((B, C, H, W), device="cuda")
    flops = 2.0 * B * H * W * 441 * C
    os.environ.pop("VSR_CORR_GENERIC", None)
    t = timed(lambda: ops.correlation(a, b, 20, 1, 20, 1, 2, 1))
    print(f"register-tiled  {t * 1e3:8.1f} us  {flops / t / 1e9:6.2f} TFLOP/s fp32")
    os.environ["VSR_CORR_GENERIC"] = "1"
    t = timed(lambda: ops.correlation(a, b, 20, 1, 20, 1, 2, 1))
    print(f"generic         {t * 1e3:8.1f} us  {flops / t / 1e9:6.2f} TFLOP/s fp32")
    os.environ.pop("VSR_CORR_GENERIC", None)
    g = torch.randn((B, 441, H, W), device="cuda")
    t = timed(lambda: ops.correlation_backward(a, b, g, 20, 1, 20, 1, 2, 1))
    print(f"backward        {t * 1e3:8.1f} us  {2 * flops / t / 1e9:6.2f} TFLOP/s fp32 (both gradients)")
    try:
        import importlib.util
        path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "correlation_cuda.so")
        spec = importlib.util.spec_from_file_location("correlation_cuda", path)
        ref = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref)
        r1, r2, out = a.new_empty(0), a.new_empty(0), a.new_empty(0)
        t = timed(lambda: ref.forward(a, b, r1, r2, out, 20, 1, 20, 1, 2, 1))
        print(f"reference (.cu) {t * 1e3:8.1f} us  {flops / t / 1e9:6.2f} TFLOP/s fp32")
    except Exception as e:  # pragma: no cover
        print("reference binary unavailable:", e)


if __name__ == "__main__":
    main()
