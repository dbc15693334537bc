"""GPU parity: the CUDA warp / projection / mask kernels (through the C ABI) against the CPU oracle
on the same seeded inputs.  Bit-exact where the arithmetic is a gather or integer; max-abs <= 1e-3
where fp32 atomics reorder sums (BASELINE.json north_star)."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from video_super_resolution_b200 import ops, synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-3  # north star: max-abs <= 1e-3 fp32 for projection / warp


def _np(t):
    return t.detach().cpu().numpy()


@pytest.mark.parametrize("shape", [(1, 3, 64, 64), (2, 3, 37, 53), (1, 2, 16, 130), (3, 5, 9, 7)])
@pytest.mark.parametrize("bilinear", [True, False])
def test_resample2d_nchw_bit_exact(shape, bilinear):
    B, C, H, W = shape
    g = torch.Generator().manual_seed(B * 1000 + W)
    img = torch.rand(shape, generator=g) * 255
    flow = (torch.rand((B, 2, H, W), generator=g) - 0.5) * 24   # reaches beyond the borders
    flow[:, :, 0, 0] = 0.5                                        # exact half-pixel tie
    flow[:, :, -1, -1] = 1000.0                                   # far out of range -> clamp
    got = _np(ops.resample2d(img.to(DEV), flow.to(DEV), 1, bilinear))
    want = orc.resample2d_nchw(img.numpy(), flow.numpy(), 1, bilinear)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("C", [3, 32, 4, 5, 1])
@pytest.mark.parametrize("bilinear", [True, False])
def test_warp_nhwc_bit_exact(C, bilinear):
    B, H, W = 2, 45, 71
    g = torch.Generator().manual_seed(C)
    src = torch.rand((B, H, W, C), generator=g) * 255
    flow = synthetic.smooth_flow(B, H, W, 8.0, seed=C) + (torch.rand((B, H, W, 2), generator=g) - 0.5)
    got = _np(ops.warp(src.to(DEV), flow.to(DEV), bilinear))
    want = orc.warp_nhwc(src.numpy(), flow.numpy(), bilinear)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("C", [3, 8])
def test_warp_fused_residual_norm(C):
    B, H, W = 2, 33, 65
    g = torch.Generator().manual_seed(10 + C)
    src = torch.rand((B, H, W, C), generator=g) * 255
    ref = torch.rand((B, H, W, C), generator=g) * 255
    flow = synthetic.smooth_flow(B, H, W, 6.0, seed=3)
    warped, norm = ops.warp(src.to(DEV), flow.to(DEV), True, ref=ref.to(DEV))
    want_w = orc.warp_nhwc(src.numpy(), flow.numpy(), True)
    want_n = orc.channelnorm_nhwc(ref.numpy() - want_w)
    assert np.array_equal(_np(warped), want_w)
    assert np.array_equal(_np(norm), want_n)


@pytest.mark.parametrize("C", [3, 32, 5])
def test_warp_fast_mode_within_tolerance(C):
    """mode 2 (pipeline default): fp32 FMA weights instead of the reference's double products;
    north star: max-abs <= 1e-3 for warps."""
    B, H, W = 2, 45, 71
    g = torch.Generator().manual_seed(40 + C)
    src = torch.rand((B, H, W, C), generator=g) * 255
    flow = synthetic.smooth_flow(B, H, W, 8.0, seed=C) + (torch.rand((B, H, W, 2), generator=g) - 0.5)
    flow[0, 0, 0] = torch.tensor([1e9, -1e9])          # beyond 2^22: takes the conversion fallback
    got = _np(ops.warp(src.to(DEV), flow.to(DEV), 2))
    want = orc.warp_nhwc(src.numpy(), flow.numpy(), True)
    assert np.abs(got - want).max() <= TOL
    ref = torch.rand((B, H, W, C), generator=g) * 255
    if C == 3:
        w2, n2 = ops.warp(src.to(DEV), flow.to(DEV), 2, ref=ref.to(DEV))
        assert np.abs(_np(n2) - orc.channelnorm_nhwc(ref.numpy() - want)).max() <= 4 * TOL


def test_huge_and_nan_flow_take_the_exact_fallback():
    B, H, W = 1, 9, 33
    g = torch.Generator().manual_seed(77)
    src = torch.rand((B, H, W, 3), generator=g) * 255
    lab = (torch.rand((B, H, W), generator=g) * 255).to(torch.uint8)
    flow = (torch.rand((B, H, W, 2), generator=g) - 0.5) * 6
    flow[0, 1, 1] = torch.tensor([5e6, -5e6])
    flow[0, 2, 2] = torch.tensor([-3e38, 3e38])
    flow[0, 3, 3] = torch.tensor([-4194304.5, 4194303.5])
    for mode in (True, False):
        assert np.array_equal(_np(ops.warp(src.to(DEV), flow.to(DEV), mode)), orc.warp_nhwc(src.numpy(), flow.numpy(), mode))
    assert np.array_equal(_np(ops.warp_labels(lab.to(DEV), flow.to(DEV))), orc.warp_labels(lab.numpy(), flow.numpy()))


def test_warp_unaligned_views_and_ragged_tail():
    # 1 pixel short of a vector multiple, and an output carved at a non-16-byte offset (through the C ABI: ops.warp
    # allocates its output aligned), which the C = 3 kernel must store element by element
    from tests.front_hooks import warp_carved
    B, H, W = 1, 17, 19
    g = torch.Generator().manual_seed(5)
    src = torch.rand((B, H, W, 3), generator=g)
    flow = (torch.rand((B, H, W, 2), generator=g) - 0.5) * 5
    ref = torch.rand((B, H, W, 3), generator=g)
    got = _np(ops.warp(src.to(DEV), flow.to(DEV)))
    assert np.array_equal(got, orc.warp_nhwc(src.numpy(), flow.numpy()))
    for mode in (0, 1, 2):
        for offset in (1, 2, 3):
            carved, norm = warp_carved(src.to(DEV), flow.to(DEV), mode, ref.to(DEV), offset_floats=offset)
            want, want_n = orc.warp_nhwc(src.numpy(), flow.numpy(), mode, ref=ref.numpy())
            assert np.array_equal(_np(carved), want) and np.array_equal(_np(norm), want_n), (mode, offset)


@pytest.mark.parametrize("shape", [(1, 64, 64), (3, 31, 45), (2, 8, 1023)])
def test_label_warp_bit_exact(shape):
    B, H, W = shape
    lab = synthetic.labels(B, H, W, seed=W)
    flow = synthetic.smooth_flow(B, H, W, 8.0, seed=H)
    flow[:, 0, 0, :] = 0.5
    got = _np(ops.warp_labels(lab.to(DEV), flow.to(DEV)))
    assert got.dtype == np.uint8
    assert np.array_equal(got, orc.warp_labels(lab.numpy(), flow.numpy()))


@pytest.mark.parametrize("shape", [(1, 3, 64, 64), (2, 2, 19, 33), (1, 7, 5, 5)])
def test_channelnorm_bit_exact(shape):
    x = torch.randn(shape, generator=torch.Generator().manual_seed(shape[1])) * 30
    got = _np(ops.channelnorm(x.to(DEV)))
    assert np.array_equal(got, orc.channelnorm_nchw(x.numpy()))


def _check_projection(flow, inv, bounds=(None,)):
    """bounds: the max_disp promises to run with (None = general scatter path; a number = shared-memory tile path,
    or its device-side fallback when the flow breaks the promise) -- every one must reproduce the oracle."""
    o_proj, o_wsum, o_count, o_hole = orc.flow_projection(flow.numpy(), inv.numpy() if inv is not None else None)
    for md in bounds:
        # "workspace: any contents" (include/vsr_b200.h): poison it, so that a path which leaves part of its bitmaps
        # unwritten cannot be rescued by what the previous call left there
        for ws in ops._WORKSPACES.values():
            ws.fill_(0xA5)
        proj, wsum, count, hole = ops.project_flow(flow.to(DEV), inv.to(DEV) if inv is not None else None, md)
        assert np.array_equal(_np(count), o_count), md        # bit-exact (north star)
        assert np.array_equal(_np(hole), o_hole), md          # bit-exact
        assert np.abs(_np(proj) - o_proj).max() <= TOL, md
        assert np.abs(_np(wsum) - o_wsum).max() <= TOL * max(1.0, float(o_wsum.max())), md
    return o_count, o_hole


@pytest.mark.parametrize("shape", [(1, 64, 64), (2, 37, 70), (1, 5, 3), (3, 130, 33)])
@pytest.mark.parametrize("weighted", [False, True])
def test_projection_smooth_flow(shape, weighted):
    B, h, w = shape
    flow = synthetic.smooth_flow(B, h, w, 8.0, seed=h)
    inv = synthetic.inv_depth(B, h, w, seed=w) if weighted else None
    # 8.0 / 3.0: the tile path (its geometry is always the 8 px one: a smaller promise this field exceeds is harmless);
    # 16.0: beyond the tile path's bound -> the general path
    _check_projection(flow, inv, bounds=(None, 8.0, 16.0, 3.0))
    # a promise the field breaks beyond 8 px: flagged on the device, the batch redone by the general path
    _check_projection(flow * 1.5, inv, bounds=(8.0,))


@pytest.mark.parametrize("shape", [(1, 200, 400), (2, 65, 193), (1, 64, 192), (3, 129, 385), (1, 80, 128), (2, 81, 130),
                                   (1, 161, 258), (2, 70, 200)])
def test_projection_tile_path_across_tile_borders(shape):
    """Sizes around the 128 x 80 tile of the shared-memory path (one tile, one tile + 1, several tiles), smooth and
    i.i.d. fields within the bound (i.i.d.: many lanes of one instruction hit the same cell -> the claim protocol)."""
    B, h, w = shape
    inv = synthetic.inv_depth(B, h, w, seed=3)
    _check_projection(synthetic.smooth_flow(B, h, w, 8.0, seed=5), inv, bounds=(8.0,))
    _check_projection(synthetic.random_flow(B, h, w, 6.0, seed=6), inv, bounds=(6.0, 7.5))
    _check_projection(synthetic.random_flow(B, h, w, 8.0, seed=7), None, bounds=(8.0,))
    _check_projection(synthetic.random_flow(B, h, w, 12.0, seed=8), None, bounds=(8.0,))      # broken promise -> redo


@pytest.mark.parametrize("weighted", [False, True])
def test_projection_collision_stress_random_flow(weighted):
    B, h, w = 2, 96, 160
    flow = synthetic.random_flow(B, h, w, 64.0, seed=1)
    inv = synthetic.inv_depth(B, h, w, seed=2) if weighted else None
    count, hole = _check_projection(flow, inv, bounds=(None, 8.0))       # 8: broken promise -> redo by the general path
    assert hole.any() and count.max() >= 4


def test_projection_zero_and_nan_depth_are_holes():
    """An inverse depth of 0 (or NaN) from a real estimator: a target whose hits carry no positive weight is a hole
    and is filled from its neighbours -- no division by zero, no NaN downstream (count stays the integer hit count)."""
    B, h, w = 1, 40, 70
    flow = torch.zeros((B, h, w, 2))
    inv = synthetic.inv_depth(B, h, w, seed=1)
    inv[0, 10:14, 20:25] = 0.0
    inv[0, 30, 60] = float("nan")
    for md in (None, 1.0):
        proj, wsum, count, hole = ops.project_flow(flow.to(DEV), inv.to(DEV), md)
        assert torch.isfinite(proj).all() and torch.isfinite(wsum).all()
        assert int(count.min()) >= 1 and bool(hole[0, 11, 21]) and bool(hole[0, 12, 23])
    _check_projection(flow, inv, bounds=(None, 1.0))


def test_projection_dense_occlusion_fill_band():
    B, h, w = 2, 72, 200
    flow, inv = synthetic.occlusion_scene(B, h, w, shift=64.0, seed=4)
    count, hole = _check_projection(flow, inv)
    assert hole.sum() > 0.05 * hole.size                   # the 64-px trailing band


def test_projection_edge_cases():
    # zero flow (duplicate clamped targets at the borders), all out of range, NaN flow, integer flow
    z = torch.zeros((1, 9, 11, 2))
    _check_projection(z, None, bounds=(None, 0.0, 2.0))
    _check_projection(torch.full((1, 6, 6, 2), 500.0), None, bounds=(None, 8.0))
    n = torch.zeros((1, 6, 7, 2))
    n[0, 2, 3, 0] = float("nan")
    _check_projection(n, None, bounds=(None, 1.0))
    i = torch.zeros((1, 12, 40, 2))
    i[..., 0] = 3.0
    i[..., 1] = -2.0
    _check_projection(i, synthetic.inv_depth(1, 12, 40, seed=9), bounds=(None, 3.0))


@pytest.mark.parametrize("shape", [(1, 1, 1), (2, 1, 40), (1, 40, 1), (1, 2, 2), (1, 17, 33), (1, 33, 65), (3, 32, 32)])
def test_projection_degenerate_shapes_and_border_hits(shape):
    """Single rows / columns, sizes straddling the 32-pixel strips, and flows that land exactly on the last row /
    column (the clamped duplicate targets = multiplicity 2 of the 2x2 box sum), half-integer and integer mixes."""
    B, h, w = shape
    g = torch.Generator().manual_seed(h * 100 + w)
    flow = torch.randint(-3, 4, (B, h, w, 2), generator=g).float()
    flow += torch.randint(0, 2, (B, h, w, 2), generator=g).float() * 0.5
    yy, xx = torch.meshgrid(torch.arange(h), torch.arange(w), indexing="ij")
    flow[:, :, -1, 0] = (w - 1 - xx[:, -1]).float()          # last column's sources stay on the last column
    flow[:, -1, :, 1] = (h - 1 - yy[-1, :]).float()          # last row's sources stay on the last row
    flow[:, 0, 0, :] = torch.tensor([float(w - 1), float(h - 1)])   # corner source -> opposite corner exactly
    for inv in (None, synthetic.inv_depth(B, h, w, seed=h + w)):
        _check_projection(flow, inv, bounds=(None, 8.0) if max(h, w) <= 8 else (None,))
    small = torch.randint(-3, 4, (B, h, w, 2), generator=g).float() * 0.5       # within +-1.5 px: the tile path
    small[:, :, -1, 0] = 0.0
    small[:, -1, :, 1] = 0.0
    _check_projection(small, synthetic.inv_depth(B, h, w, seed=1), bounds=(1.5, 2.0))


def test_projection_full_size_properties():
    # C3 size (1080p): size-independent properties instead of the slow CPU oracle
    B, h, w = 2, 1080, 1920            # 420 tiles: the tile path (a single image's 210 tiles take the general path)
    flow = synthetic.smooth_flow(B, h, w, 8.0, seed=0).to(DEV)
    inv = synthetic.inv_depth(B, h, w, seed=1).to(DEV)
    proj, wsum, count, hole = ops.project_flow(flow, inv, 8.0)
    x2 = torch.arange(w, device=DEV).view(1, 1, w) + flow[..., 0]
    y2 = torch.arange(h, device=DEV).view(1, h, 1) + flow[..., 1]
    valid = (x2 >= 0) & (x2 <= w - 1) & (y2 >= 0) & (y2 <= h - 1)
    assert int(count.sum()) == 4 * int(valid.sum())          # every valid source hits 4 targets
    assert torch.equal(hole.bool(), count == 0)
    wtot = (inv * valid).sum().item() * 4
    assert abs(wsum.sum().item() - wtot) <= 1e-4 * wtot      # linearity: total weight conserved
    assert proj.abs().max().item() <= 8.0 + 1e-3             # a weighted mean of |flow| <= 8
    # idempotent / deterministic integers
    proj2, wsum2, count2, hole2 = ops.project_flow(flow, inv)          # the general path agrees with the tile path
    assert torch.equal(count, count2) and torch.equal(hole, hole2)
    assert (proj - proj2).abs().max().item() <= 1e-3 and (wsum - wsum2).abs().max().item() <= 1e-3


def test_vos_threshold_and_mask_fill_bit_exact():
    la, lb = synthetic.logits(67, 129, seed=3)
    mask = ops.vos_threshold(la.to(DEV), lb.to(DEV))
    want = orc.vos_threshold(la.numpy(), lb.numpy())
    assert np.array_equal(_np(mask), want)
    assert 0 < want.mean() < 1
    img = torch.rand((3, 67, 129), generator=torch.Generator().manual_seed(1)) * 255
    got = _np(ops.mask_fill(img.to(DEV), mask))
    assert np.array_equal(got, orc.mask_fill(img.numpy(), want))


def test_golden_vos_fixture_on_gpu(golden_dir):
    import os
    z = np.load(os.path.join(golden_dir, "vos_mask.npz"))
    la = torch.from_numpy(z["logits"])
    mask = ops.vos_threshold(la[0, 0].contiguous().to(DEV), la[1, 0].contiguous().to(DEV))
    assert np.array_equal(_np(mask).astype(np.float32), z["mask"])
    filled = ops.mask_fill(torch.from_numpy(z["image"]).to(DEV), mask)
    assert np.array_equal(_np(filled), z["filled"])


def test_launches_are_counted():
    from video_super_resolution_b200 import _lib
    _lib.launch_count_reset()
    x = torch.zeros((1, 3, 8, 8), device=DEV)
    ops.channelnorm(x)
    assert _lib.launch_count() == 1


def test_projection_random_shapes_and_fields_against_oracle():
    """Seeded sweep over shapes (around the tile / block / strip sizes, odd and even widths), batch sizes, weighted and
    unweighted, smooth / i.i.d. / mixed fields, kept and broken promises -- every path must reproduce the oracle
    (count / hole bit for bit), starting from a poisoned workspace."""
    rng = np.random.default_rng(1234)
    for it in range(24):
        B = int(rng.integers(1, 4))
        h = int(rng.choice([1, 7, 16, 31, 47, 79, 80, 81, 97, 130, 161]))
        w = int(rng.choice([2, 15, 16, 34, 126, 128, 130, 160, 257, 300]))
        kind = it % 4
        mag = float(rng.choice([0.5, 3.0, 8.0]))
        if kind == 0:
            flow = synthetic.smooth_flow(B, h, w, mag, seed=it)
        elif kind == 1:
            flow = synthetic.random_flow(B, h, w, mag, seed=it)
        elif kind == 2:       # half-integer steps: many exact cell-border and image-border hits, many collisions
            flow = torch.from_numpy(rng.integers(-16, 17, size=(B, h, w, 2)).astype(np.float32) * 0.5)
        else:                 # smooth field with a few far movers: the promise of 8 px is broken
            flow = synthetic.smooth_flow(B, h, w, 6.0, seed=it)
            flow[:, h // 2, :: max(w // 5, 1), 0] = 23.0
        inv = synthetic.inv_depth(B, h, w, seed=100 + it) if it % 3 else None
        _check_projection(flow, inv, bounds=(8.0, None))


def test_projection_tile_path_needs_aligned_pixel_pairs():
    """The tile path loads two pixels at a time (16-byte flow, 8-byte depth loads): a flow that starts 8 bytes into a
    16-byte line or a depth map that starts 4 bytes into an 8-byte word takes the general path -- same results."""
    B, h, w = 2, 90, 140
    flow = synthetic.smooth_flow(B, h, w, 6.0, seed=3)
    inv = synthetic.inv_depth(B, h, w, seed=4)
    want = orc.flow_projection(flow.numpy(), inv.numpy())
    fbuf = torch.empty(flow.numel() + 2, device=DEV)
    dbuf = torch.empty(inv.numel() + 1, device=DEV)
    f_off = fbuf[2:].view(B, h, w, 2)
    d_off = dbuf[1:].view(B, h, w)
    f_off.copy_(flow)
    d_off.copy_(inv)
    assert f_off.data_ptr() % 16 == 8 and d_off.data_ptr() % 8 == 4
    for fl, dp in ((f_off, inv.to(DEV)), (flow.to(DEV), d_off), (f_off, d_off)):
        proj, wsum, count, hole = ops.project_flow(fl, dp, 8.0)
        assert np.array_equal(_np(count), want[2]) and np.array_equal(_np(hole), want[3])
        assert np.abs(_np(proj) - want[0]).max() <= TOL and np.abs(_np(wsum) - want[1]).max() <= TOL * max(1.0, float(want[1].max()))
