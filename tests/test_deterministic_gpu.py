"""The deterministic flow projection and Resample2d input gradient: bit-identical to the CPU restatement
(oracle.or_flow_projection, oracle.or_resample2d_backward), selected by `deterministic=True` or by
torch.use_deterministic_algorithms(True).  The last tests check the host side without a GPU."""
import contextlib

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from video_super_resolution_b200 import _lib, ops, synthetic as syn

DEV = "cuda:0"
gpu = pytest.mark.gpu


@contextlib.contextmanager
def _torch_deterministic():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def _field(kind, B, h, w, seed):
    """(flow, inv_depth) of one of C3's three flow fields."""
    if kind == "smooth8":
        return syn.smooth_flow(B, h, w, 8.0, seed=seed), syn.inv_depth(B, h, w, seed=seed + 1)
    if kind == "iid64":
        return syn.random_flow(B, h, w, 64.0, seed=seed), syn.inv_depth(B, h, w, seed=seed + 1)
    return syn.occlusion_scene(B, h, w, 64.0, seed=seed)


def _project(flow, inv):
    """ops.project_flow(deterministic=True) with the cached workspace poisoned first (it may hold anything)."""
    B, h, w, _ = flow.shape
    nbytes = int(_lib.lib().vsr_flow_projection_deterministic_workspace_bytes(B, h, w))
    with torch.cuda.device(DEV):
        ops._workspace(nbytes, torch.device(DEV)).fill_(0xA5)
    got = ops.project_flow(flow.to(DEV), inv.to(DEV) if inv is not None else None, deterministic=True)
    return [t.cpu().numpy() for t in got]


def _assert_projection_equal(flow, inv):
    got = _project(flow, inv)
    want = orc.flow_projection(flow.numpy(), inv.numpy() if inv is not None else None)
    for name, g, e in zip(("proj", "wsum", "count", "hole"), got, want):
        assert g.dtype == e.dtype and np.array_equal(g, e), (name, np.argwhere(g != e)[:5])


@gpu
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("kind", ["smooth8", "iid64", "occlusion"])
@pytest.mark.parametrize("B,h,w", [(1, 1, 1), (1, 1, 7), (1, 5, 3), (2, 37, 53), (3, 130, 33)])
def test_projection_bit_identical_to_oracle(B, h, w, kind, weighted):
    flow, inv = _field(kind, B, h, w, seed=B * 100 + h + w)
    _assert_projection_equal(flow, inv if weighted else None)


@gpu
@pytest.mark.parametrize("weighted", [False, True])
def test_projection_edge_values(weighted):
    """NaN flow, zero and NaN inverse depth, and sources that land exactly on the last column / row (the clamped
    duplicate targets)."""
    B, h, w = 2, 37, 53
    flow, inv = _field("iid64", B, h, w, seed=11)
    g = torch.Generator().manual_seed(12)
    pick = lambda k: torch.randint(0, h * w, (k,), generator=g)
    fl, dp = flow.view(B, h * w, 2), inv.view(B, h * w)
    fl[0, pick(40), 0] = float("nan")
    fl[1, pick(40), 1] = float("nan")
    dp[:, pick(60)] = 0.0
    dp[:, pick(30)] = float("nan")
    ys, xs = torch.meshgrid(torch.arange(h, dtype=torch.float32), torch.arange(w, dtype=torch.float32), indexing="ij")
    on_col, on_row = pick(80), pick(80)
    fl[:, on_col, 0] = (w - 1) - xs.reshape(-1)[on_col]
    fl[:, on_row, 1] = (h - 1) - ys.reshape(-1)[on_row]
    corner = pick(10)
    fl[:, corner, 0] = (w - 1) - xs.reshape(-1)[corner]
    fl[:, corner, 1] = (h - 1) - ys.reshape(-1)[corner]
    _assert_projection_equal(flow, inv if weighted else None)


@gpu
@pytest.mark.parametrize("kind", ["smooth8", "iid64", "occlusion"])
def test_projection_1080p_c3_fields(kind):
    flow, inv = _field(kind, 2, 1080, 1920, seed=21)
    _assert_projection_equal(flow, None)
    _assert_projection_equal(flow, inv)


@gpu
def test_projection_skew_every_source_in_one_cell():
    h = w = 256
    ys, xs = torch.meshgrid(torch.arange(h, dtype=torch.float32), torch.arange(w, dtype=torch.float32), indexing="ij")
    flow = torch.stack((100.5 - xs, 60.25 - ys), dim=-1)[None].contiguous()
    inv = syn.inv_depth(1, h, w, seed=3)
    _assert_projection_equal(flow, inv)


def _resample_inputs(B, C, H, W, seed, mag=4.0):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand((B, C, H, W), generator=g) * 255
    flow = (torch.rand((B, 2, H, W), generator=g) * 2 - 1) * mag
    go = torch.randn((B, C, H, W), generator=g)
    return x, flow, go


@gpu
@pytest.mark.parametrize("C", [1, 3, 32])
def test_resample2d_backward_deterministic(C):
    x, flow, go = _resample_inputs(2, C, 37, 53, seed=C)
    flow[0, :, :3, :] *= 20          # some samples outside the image: clamped taps
    want1, _ = orc.resample2d_backward(x.numpy(), flow.numpy(), go.numpy())
    xd, fd, gd = x.to(DEV), flow.to(DEV), go.to(DEV)
    g1, g2 = ops.resample2d_backward(xd, fd, gd, deterministic=True)
    _, g2_atomic = ops.resample2d_backward(xd, fd, gd, deterministic=False)
    assert np.array_equal(g1.cpu().numpy(), want1)
    assert torch.equal(g2, g2_atomic)
    # every element is written: a grad_input1 full of NaN on entry gives the same result
    B, C_, H, W = x.shape
    L = _lib.lib()
    ws = torch.full((int(L.vsr_resample2d_backward_deterministic_workspace_bytes(B, H, W)),), 0xA5, dtype=torch.uint8,
                    device=DEV)
    g1n, g2n = torch.full_like(xd, float("nan")), torch.empty_like(fd)
    rc = L.vsr_resample2d_backward_deterministic(xd.data_ptr(), fd.data_ptr(), gd.data_ptr(), g1n.data_ptr(),
                                                 g2n.data_ptr(), B, C_, H, W, 1, 1, ws.data_ptr(), ws.numel(),
                                                 torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    assert torch.equal(g1n, g1) and torch.equal(g2n, g2)
    rc = L.vsr_resample2d_backward_deterministic(xd.data_ptr(), fd.data_ptr(), gd.data_ptr(), g1n.data_ptr(),
                                                 g2n.data_ptr(), B, C_, H, W, 2, 1, ws.data_ptr(), ws.numel(),
                                                 torch.cuda.current_stream().cuda_stream)
    assert rc == 2                   # VSR_ERR_UNSUPPORTED: kernel_size 2
    with pytest.raises(_lib.VsrError, match="unsupported"):
        ops.resample2d_backward(xd, fd, gd, kernel_size=2, deterministic=True)


@gpu
def test_resample2d_backward_skew_every_sample_outside():
    """Every sample lands outside the image: the clamped taps send the whole image to one border pixel, which sums
    them in sequence."""
    x, flow, go = _resample_inputs(1, 3, 256, 256, seed=5)
    flow.fill_(1000.0)
    flow[0, 1] += torch.rand((256, 256), generator=torch.Generator().manual_seed(6))
    want1, _ = orc.resample2d_backward(x.numpy(), flow.numpy(), go.numpy())
    g1, _ = ops.resample2d_backward(x.to(DEV), flow.to(DEV), go.to(DEV), deterministic=True)
    assert np.array_equal(g1.cpu().numpy(), want1)


@gpu
def test_torch_deterministic_flag_selects_the_deterministic_paths():
    from video_super_resolution_b200.integration import resample2d_cuda as stub
    B, h, w = 2, 130, 170
    flow = syn.random_flow(B, h, w, 64.0, seed=31)
    want = orc.flow_projection(flow.numpy(), None)
    fast = ops.project_flow(flow.to(DEV), deterministic=False)
    # fp32 sums in arrival order against the oracle's fp64 sums: the default path differs somewhere, so the checks
    # below are meaningful
    assert not np.array_equal(fast[0].cpu().numpy(), want[0])
    x, rflow, go = _resample_inputs(2, 3, 40, 60, seed=32, mag=64.0)
    want1, _ = orc.resample2d_backward(x.numpy(), rflow.numpy(), go.numpy())
    with _torch_deterministic():
        got = ops.project_flow(flow.to(DEV))
        for g, e in zip(got, want):
            assert np.array_equal(g.cpu().numpy(), e)
        xd, fd, gd = x.to(DEV), rflow.to(DEV), go.to(DEV)
        g1, g2 = torch.zeros_like(xd), torch.zeros_like(fd)
        assert stub.backward(xd, fd, gd, g1, g2, 1, True) == 1
        assert np.array_equal(g1.cpu().numpy(), want1)
        from video_super_resolution_b200.my_packages.FlowProjection.networks.resample2d_package.resample2d import \
            Resample2d
        xr = xd.clone().requires_grad_(True)
        Resample2d()(xr, fd).backward(gd)
        assert np.array_equal(xr.grad.cpu().numpy(), want1)
    assert not torch.are_deterministic_algorithms_enabled()


def _pipeline(T, h, w, seed):
    from oracle import srfbn_oracle as so
    from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
    from video_super_resolution_b200.pipeline import WarpFusePipeline
    M = 3 * T - 1
    sr = SRProjectionModule(num_maps=M)
    sr.load_state_dict(so.init_state_dict(num_maps=M, seed=seed, gain=2.3))
    pipe = WarpFusePipeline(T, h, w, sr, 4, device=DEV, max_disp=None)
    la, lb = syn.logits(h, w, seed=seed + 3)
    args = (syn.frames(T, h, w, seed=seed), syn.random_flow(T - 1, h, w, 64.0, seed=seed + 1),
            syn.inv_depth(T - 1, h, w, seed=seed + 2), la, lb)
    return pipe, args


@gpu
@pytest.mark.parametrize("T,h,w", [(3, 32, 48), (7, 270, 480)])
def test_pipeline_under_the_flag_is_bit_exact_and_repeatable(T, h, w):
    """WarpFusePipeline(max_disp=None) on +-64 px flow under torch.use_deterministic_algorithms(True): the label warp
    equals the oracle's warp of the oracle's projected flow with no tolerance, and two full steps (conv stack included)
    give byte-identical frames."""
    pipe, args = _pipeline(T, h, w, seed=T)
    dargs = [t.to(DEV) for t in args]
    _, want = orc.warp_fuse_front(*[t.numpy() for t in args], threads=8)
    with _torch_deterministic():
        r = pipe.project_and_warp(*dargs)
        for k in ("proj_flow", "count_flow", "hole_flow", "proj_depth", "wsum", "count_depth", "hole_depth",
                  "mask_warped"):
            assert np.array_equal(r[k].cpu().numpy(), want[k]), k
        frames = []
        for _ in range(2):
            u8 = torch.zeros((4 * h, 4 * w, 3), dtype=torch.uint8, device=DEV)
            pipe.step(*dargs, out_u8=u8, want_f32=False)
            frames.append(u8.cpu())
    assert torch.equal(frames[0], frames[1]) and int(frames[0].max()) > 0


# ---- host side, no GPU needed ----

def test_deterministic_workspace_sizes_without_gpu():
    L = _lib.lib()
    P = 1080 * 1920
    # four key / value arrays and the per-cell ranges (4 B each per pixel), histograms, bitmaps, hole list: one image
    n = L.vsr_flow_projection_deterministic_workspace_bytes(8, 1080, 1920)
    assert 5 * 4 * P <= n < 5 * 4 * P + (8 << 20)
    assert n == L.vsr_flow_projection_deterministic_workspace_bytes(1, 1080, 1920)
    m = L.vsr_resample2d_backward_deterministic_workspace_bytes(2, 1080, 1920)
    assert 5 * 4 * 2 * P <= m < 5 * 4 * 2 * P + (16 << 20)
    for bad in ((0, 4, 4), (1, 0, 4), (1, 4, -1)):
        assert L.vsr_flow_projection_deterministic_workspace_bytes(*bad) == 0
        assert L.vsr_resample2d_backward_deterministic_workspace_bytes(*bad) == 0


def test_deterministic_argument_errors_without_gpu():
    L = _lib.lib()
    big = 1 << 40
    # projection: null pointers / sizes, unsupported size, small workspace, misaligned workspace
    assert L.vsr_flow_projection_forward_deterministic(None, None, 16, None, 16, 16, 16, big, 1, 4, 4, None) == 1
    assert L.vsr_flow_projection_forward_deterministic(16, None, 16, None, 16, 16, 16, big, 0, 4, 4, None) == 1
    assert L.vsr_flow_projection_forward_deterministic(16, None, 16, None, 16, 16, 16, big, 1, 32768, 32769, None) == 2
    assert L.vsr_flow_projection_forward_deterministic(16, None, 16, None, 16, 16, 16, 64, 1, 4, 4, None) == 3
    assert L.vsr_flow_projection_forward_deterministic(16, None, 16, None, 16, 16, 20, big, 1, 4, 4, None) == 1
    # resample2d backward: null pointers, kernel_size, 32-bit bound, small workspace
    assert L.vsr_resample2d_backward_deterministic(16, 16, 16, None, 16, 1, 3, 4, 4, 1, 1, 16, big, None) == 1
    assert L.vsr_resample2d_backward_deterministic(16, 16, 16, 16, 16, 1, 3, 4, 4, 1, 1, None, big, None) == 1
    assert L.vsr_resample2d_backward_deterministic(16, 16, 16, 16, 16, 1, 3, 4, 4, 2, 1, 16, big, None) == 2
    assert L.vsr_resample2d_backward_deterministic(16, 16, 16, 16, 16, 4, 1, 32768, 32768, 1, 1, 16, big, None) == 2
    assert L.vsr_resample2d_backward_deterministic(16, 16, 16, 16, 16, 1, 3, 4, 4, 1, 1, 16, 64, None) == 3


def test_deterministic_ops_refuse_cpu_tensors():
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.project_flow(torch.zeros(1, 4, 4, 2), deterministic=True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.resample2d_backward(torch.zeros(1, 3, 4, 4), torch.zeros(1, 2, 4, 4), torch.zeros(1, 3, 4, 4),
                                deterministic=True)
