"""GPU tests of BASELINE.json's configurations (C1 .. C5) at their full sizes through properties that do not need the CPU
oracle at that size, plus direct oracle comparisons where the C oracle is fast enough."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from video_super_resolution_b200 import ops, synthetic as syn
from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
from video_super_resolution_b200.network.video_super_resolution import VSR
from video_super_resolution_b200.pipeline import shard_windows

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def test_c1_single_pair_64x64_plumbing():
    """C1: one synthetic frame pair 64x64, random flow + depth: FlowProjection, DepthProjection and the bilinear
    warp along the projected flow, GPU (through the C ABI) against the CPU oracle."""
    h = w = 64
    flow = syn.random_flow(1, h, w, 6.0, seed=1)
    inv = syn.inv_depth(1, h, w, seed=2)
    frame = syn.frames(1, h, w, seed=3)
    for d in (None, inv):
        if d is None:
            proj, wsum, count, hole = ops.project_flow(flow.to(DEV))
        else:
            proj, wsum, count, hole = ops.project_depth_flow(flow.to(DEV), d.to(DEV))
        o_proj, o_wsum, o_count, o_hole = orc.flow_projection(flow.numpy(), None if d is None else d.numpy())
        assert np.array_equal(count.cpu().numpy(), o_count) and np.array_equal(hole.cpu().numpy(), o_hole)
        assert np.abs(proj.cpu().numpy() - o_proj).max() <= 1e-3
        warped = ops.warp(frame.to(DEV), proj, True)                     # reference arithmetic, bit for bit
        assert np.array_equal(warped.cpu().numpy(), orc.warp_nhwc(frame.numpy(), proj.cpu().numpy(), True))


def test_c3_large_motion_occlusion_1080p_against_oracle():
    """C3: 1080p, +-64 px, dense occlusion, DepthProjection splat: count / hole bit-exact, sums <= 1e-3."""
    h, w = 1080, 1920
    flow, inv = syn.occlusion_scene(1, h, w, shift=64.0, seed=5)
    flow = flow + syn.random_flow(1, h, w, 0.75, seed=6)          # break the integer-flow symmetry
    proj, wsum, count, hole = ops.project_depth_flow(flow.to(DEV), inv.to(DEV))
    o_proj, o_wsum, o_count, o_hole = orc.flow_projection(flow.numpy(), inv.numpy())
    assert np.array_equal(count.cpu().numpy(), o_count)
    assert np.array_equal(hole.cpu().numpy(), o_hole)
    assert np.abs(proj.cpu().numpy() - o_proj).max() <= 1e-3
    assert np.abs(wsum.cpu().numpy() - o_wsum).max() <= 1e-3 * max(1.0, float(o_wsum.max()))
    assert o_hole.mean() > 0.01 and o_count.max() >= 6


def test_c3_random_64px_1080p_against_oracle():
    h, w = 1080, 1920
    flow = syn.random_flow(1, h, w, 64.0, seed=8)
    inv = syn.inv_depth(1, h, w, seed=9)
    proj, wsum, count, hole = ops.project_depth_flow(flow.to(DEV), inv.to(DEV))
    o_proj, o_wsum, o_count, o_hole = orc.flow_projection(flow.numpy(), inv.numpy())
    assert np.array_equal(count.cpu().numpy(), o_count)
    assert np.array_equal(hole.cpu().numpy(), o_hole)
    assert np.abs(proj.cpu().numpy() - o_proj).max() <= 1e-3


def test_c2_conv_stack_full_size_is_deterministic_and_tiling_consistent():
    """C2 (M=20, 270x480 -> 1080x1920): (1) two runs give identical bits (no atomics in the stack);
    (2) the output over an interior window equals the output of the same network run on a crop of the
    input that contains the window's receptive field -- a check of every tile / ring / edge rule at
    full size that needs no CPU oracle; (3) chunked plans under workspace caps give the same bits."""
    M, h, w = 20, 270, 480
    torch.manual_seed(0)
    sr = SRProjectionModule(num_maps=M)
    with torch.no_grad():
        for n, p in sr.named_parameters():
            if n.endswith(".0.weight") and not n.startswith(("sub_mean", "add_mean")):
                p.mul_(2.3)
    x = (torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(1)) * 255).to(DEV)
    y1 = sr(x)
    y2 = sr(x)
    assert torch.isfinite(y1).all()
    assert torch.equal(y1, y2)
    # receptive field: 3 steps x 6 groups x (deconv +-1, conv +-1 LR px) + 3x3 convs < 48 LR pixels
    y0, x0, ch, cw, m = 64, 128, 128, 192, 48
    yc = sr(x[:, :, y0:y0 + ch, x0:x0 + cw].contiguous())
    a = y1[:, :, 4 * (y0 + m):4 * (y0 + ch - m), 4 * (x0 + m):4 * (x0 + cw - m)]
    b = yc[:, :, 4 * m:4 * (ch - m), 4 * m:4 * (cw - m)]
    assert a.shape == b.shape and a.numel() > 0
    assert (a - b).abs().max().item() <= 1e-2 * (a.abs().mean().item() + 1.0)
    # (3) the same frame under workspace caps: 10, 5 and 4 maps per sweep over the layer list instead of 20, bit for
    # bit (every chunk runs the merged up-down kernel of groups 3-5 on its own slice of the maps)
    import gc
    full = sr._plans[(M, h, w, 0)]["workspace"].numel()
    sd = {k: v.detach().clone() for k, v in sr.state_dict().items()}
    del sr, y2, yc, a, b
    gc.collect()
    torch.cuda.empty_cache()
    for frac, chunk in ((0.55, 10), (0.3, 5), (0.23, 4)):
        cap = SRProjectionModule(num_maps=M, workspace_cap_bytes=int(full * frac))
        cap.load_state_dict(sd)
        y3 = cap(x)
        ent = next(iter(cap._plans.values()))
        assert ent["chunk_maps"] == chunk and ent["workspace"].numel() <= full * frac, (frac, ent["chunk_maps"])
        assert torch.equal(y3, y1), frac
        del cap, y3, ent
        gc.collect()
        torch.cuda.empty_cache()


def _oracle_maps_on_gpu(x, sd, steps, scale):
    """oracle/srfbn_oracle.forward_maps as the CHECKER, on the GPU in fp32 (TF32 off: cuDNN / cuBLAS fp32 FMA),
    one map at a time so that the six HR feature maps and their concats stay small."""
    from oracle import srfbn_oracle as so
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        sdc = {k: v.to(DEV, torch.float32) for k, v in sd.items()}
        with torch.no_grad():
            return torch.cat([so.forward_maps(x[m:m + 1], sdc, num_steps=steps, upscale=scale) for m in range(x.shape[0])])
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _psnr255(a, b):
    import math
    mse = ((a.double() - b.double()) ** 2).mean().item()
    return 10 * math.log10(255.0 ** 2 / max(mse, 1e-20))


@pytest.mark.parametrize("name,M,h,w,scale", [("C2", 20, 270, 480, 4), ("C4crop", 14, 264, 328, 2)])
def test_conv_stack_full_size_against_fp32_oracle(name, M, h, w, scale):
    """The conv stack at C2's FULL size (M=20, 270x480 -> 1080x1920; tile-walk carries, the (h+1)x(w+1) block ring,
    2.67 GB strides -- what a 24x40 case cannot reach) and on a >= 256x256 LR crop of C4 (x2, M=14) against the fp32
    oracle: per-map PSNR > 50 dB and the north star's PSNR delta <= 0.05 dB against a common target ~35 dB away.
    Same asserts as tests/test_srfbn_gpu.py::test_full_stack_against_oracle."""
    import gc
    from oracle import srfbn_oracle as so
    gc.collect()
    torch.cuda.empty_cache()
    sd = so.init_state_dict(num_maps=M, seed=11, gain=2.3, upscale=scale)
    gs = torch.Generator().manual_seed(99)
    for k in sd:
        if k.endswith(".1.weight"):
            sd[k] = torch.rand(1, generator=gs) * 0.4 + 0.05             # distinct slopes: a mixed-up layer shows
    mod = SRProjectionModule(num_maps=M, upscale_factor=scale)
    mod.load_state_dict(sd)
    x = (torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(5)) * 255).to(DEV)
    got = mod.premix(x)
    want = _oracle_maps_on_gpu(x, sd, 3, scale)
    assert got.shape == want.shape == (M, 3, scale * h, scale * w) and torch.isfinite(got).all()
    skip = torch.nn.functional.interpolate(x, scale_factor=scale, mode="bilinear", align_corners=False)
    assert (want - skip).abs().mean().item() > 0.05                        # the conv branch carries signal
    noise = torch.randn(want.shape[1:], generator=torch.Generator().manual_seed(6)).to(DEV) * 4.5
    worst_psnr, worst_delta = 1e9, 0.0
    for m in range(M):                                                     # per map
        p = _psnr255(got[m], want[m])
        target = want[m] + noise
        d = abs(_psnr255(got[m], target) - _psnr255(want[m], target))
        worst_psnr, worst_delta = min(worst_psnr, p), max(worst_delta, d)
    assert worst_psnr > 50.0, f"{name}: worst per-map PSNR {worst_psnr:.2f} dB"
    assert worst_delta <= 0.05, f"{name}: worst PSNR delta {worst_delta:.4f} dB"
    # no tile / ring / edge artefact hides in the mean: the largest single-pixel error stays at the BF16 scale
    assert (got - want).abs().max().item() <= 0.02 * (want.abs().mean().item() + 1.0) + 0.5
    del mod, got, want, x, skip
    gc.collect()
    torch.cuda.empty_cache()


def test_c5_window_sharding_matches_single_run_at_shard_starts():
    """C5 semantics at small size: a sequence processed in one go vs in two shards.  Within a shard the
    estimate of window k feeds window k+1 (main.py:199-203); a shard starts with estimated_image=None
    (main.py:196), so shard 2's first window equals a single run restarted at that window."""
    T, h, w, n_frames = 3, 24, 32, 7
    g = torch.Generator().manual_seed(3)
    frames = (torch.rand((n_frames, h, w, 3), generator=g) * 255).to(DEV)
    flows = syn.smooth_flow(n_frames - 1, h, w, 3.0, seed=4).to(DEV)
    inv = syn.inv_depth(n_frames - 1, h, w, seed=5).to(DEV)
    la, lb = syn.logits(h, w, seed=6)
    la, lb = la.to(DEV), lb.to(DEV)
    torch.manual_seed(1)
    vsr = VSR(window=T)
    n_win = n_frames - T + 1

    def run(windows, est=None):
        outs = []
        for k in windows:
            out = vsr.forward_geometry(frames[k:k + T], flows[k:k + T - 1], inv[k:k + T - 1], la, lb, est)
            est = out
            outs.append(out)
        return outs

    whole = run(range(n_win))
    shards = [run(shard_windows(n_win, 2, r)) for r in range(2)]
    assert len(shards[0]) + len(shards[1]) == n_win
    for a, b in zip(whole[:len(shards[0])], shards[0]):
        assert torch.equal(a, b)                                  # shard 0 == the single run
    k1 = list(shard_windows(n_win, 2, 1))[0]
    restart = run([k1])[0]
    assert torch.equal(shards[1][0], restart)                     # recurrence reset at the shard start
    assert not torch.equal(shards[1][0], whole[k1])               # ... which is a real difference


def test_c4_2x_4k_conv_stack_full_size_is_deterministic_and_tiling_consistent():
    """C4 (2x, 1080x1920 -> 2160x3840, T=5 => M=14, one window per GPU): SRFBN's k6 s2 p2 geometry (the
    reference has none, SURVEY.md 8 a6).  Same two properties as C2: bit-identical reruns and equality with
    a crop run that contains the receptive field.  ~89 GB of workspace: sized for the 180 GB part."""
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    M, h, w = 14, 1080, 1920
    torch.manual_seed(0)
    sr = SRProjectionModule(num_maps=M, upscale_factor=2)
    with torch.no_grad():
        for n, p in sr.named_parameters():
            if n.endswith(".0.weight") and not n.startswith(("sub_mean", "add_mean")):
                p.mul_(2.3)
    x = (torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(1)) * 255).to(DEV)
    y1 = sr(x)
    y2 = sr(x)
    assert y1.shape == (1, 3, 2 * h, 2 * w)
    assert torch.isfinite(y1).all()
    assert torch.equal(y1, y2)
    # receptive field: 3 steps x 6 groups x (deconv +-1, conv +-2 LR px) + 3x3 convs < 64 LR pixels
    y0, x0, ch, cw, m = 400, 800, 160, 224, 64
    yc = sr(x[:, :, y0:y0 + ch, x0:x0 + cw].contiguous())
    a = y1[:, :, 2 * (y0 + m):2 * (y0 + ch - m), 2 * (x0 + m):2 * (x0 + cw - m)]
    b = yc[:, :, 2 * m:2 * (ch - m), 2 * m:2 * (cw - m)]
    assert a.shape == b.shape and a.numel() > 0
    assert (a - b).abs().max().item() <= 1e-2 * (a.abs().mean().item() + 1.0)
    del sr, y2, yc
    gc.collect()
    torch.cuda.empty_cache()
    # the same frame under a 40 GB workspace cap: 2 maps at a time instead of 14 (89 GB), bit-identical
    cap = SRProjectionModule(num_maps=M, upscale_factor=2, workspace_cap_bytes=40 << 30)
    torch.manual_seed(0)
    fresh = SRProjectionModule(num_maps=M, upscale_factor=2)
    with torch.no_grad():
        for n, p in fresh.named_parameters():
            if n.endswith(".0.weight") and not n.startswith(("sub_mean", "add_mean")):
                p.mul_(2.3)
    cap.load_state_dict(fresh.state_dict())
    y3 = cap(x)
    ent = next(iter(cap._plans.values()))
    assert ent["chunk_maps"] == 2 and ent["workspace"].numel() <= 40 << 30
    assert torch.equal(y3, y1)
    del cap, fresh, y1, y3, x
    gc.collect()
    torch.cuda.empty_cache()


def test_unsupported_geometry_is_rejected_loudly():
    """x3 / x8 exist in SRFBN but neither in the reference nor in BASELINE's configs: say so."""
    with pytest.raises(NotImplementedError):
        SRProjectionModule(upscale_factor=3)
