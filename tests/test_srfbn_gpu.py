"""GPU parity of the fusion / upsampling convolutions (tcgen05 implicit GEMM, BF16 in / FP32
accumulate) against torch.nn.functional fp32 -- the reference's own arithmetic provider for these
layers (blocks.py:16,34; SRProjectionModule.py:126-131) -- layer by layer and end to end against
oracle/srfbn_oracle.py (intended dense-concat dataflow, SURVEY.md Appendix C).

Tolerances: one layer fed BF16-rounded inputs/weights differs from fp32 math only by accumulation
order and the BF16 rounding of the output (rel 2^-8); whole stack: PSNR delta <= 0.05 dB
(BASELINE.json north_star), measured against a target placed ~35 dB from the fp32 output.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import srfbn_oracle as so
from tests import srfbn_hooks as hk
from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _bf(t):
    return t.to(torch.bfloat16)


# Largest fraction of a layer's BF16 outputs that may differ at all from the restatement fed the same BF16 operands
# (hk.faithful_bf16): a difference needs the fp32 accumulation error to cross a BF16 rounding boundary.  About 4x the
# worst measured on a B200: 0.044 % for the one-GEMM layers, 0.57 % for the fused down kernels, whose on-chip H (and U)
# rounds once more before the strided conv.
_MAX_DIFF_FRAC = 0.002
_MAX_DIFF_FRAC_FUSED = 0.025


def _d(t):
    return t.to(DEV, torch.float64)


def _close(got, want, what):
    got = got.float().cpu()
    want = want.float().cpu()
    assert torch.isfinite(got).all(), f"{what}: non-finite output"
    err = (got - want).abs()
    tol = 0.02 * want.abs() + 0.02 * want.abs().mean() + 1e-3
    bad = (err > tol).sum().item()
    assert bad == 0, f"{what}: {bad}/{err.numel()} outside tolerance, max err {err.max():.4g} (ref max {want.abs().max():.4g})"


@pytest.mark.parametrize("rows,K", [(128, 32), (1000, 64), (129, 96), (4096 + 77, 192), (300, 224)])
def test_pointwise_layer(rows, K):
    g = torch.Generator().manual_seed(rows + K)
    x = _bf(torch.randn((rows, K), generator=g))
    w = _bf(torch.randn((32, K), generator=g) / math.sqrt(K)).float()
    b = torch.randn(32, generator=g) * 0.1
    got = hk.pointwise(x.to(DEV), w, b, 0.2)
    want = F.prelu(x.float() @ w.t() + b, torch.tensor([0.2]))
    _close(got, want, f"pointwise rows={rows} K={K}")
    pre, absdot = _d(x) @ _d(w).t() + _d(b), _d(x).abs() @ _d(w).abs().t() + _d(b).abs()
    want = hk.act(pre, 0.2)
    hk.faithful_bf16(got, want, absdot, f"pointwise rows={rows} K={K} faithful", max_frac=_MAX_DIFF_FRAC,
                     ulps=hk.ulps(want))


@pytest.mark.parametrize("slope", [0.0, 1.0, 1.7, -0.3])
def test_pointwise_prelu_slope_forms(slope):
    """The packed-BF16 PReLU picks max/min/general forms by the (per-layer) slope."""
    g = torch.Generator().manual_seed(3)
    x = _bf(torch.randn((777, 64), generator=g))
    w = _bf(torch.randn((32, 64), generator=g) / 8).float()
    b = torch.randn(32, generator=g) * 0.1
    got = hk.pointwise(x.to(DEV), w, b, slope)
    want = F.prelu(x.float() @ w.t() + b, torch.tensor([slope]))
    _close(got, want, f"pointwise slope={slope}")
    pre, absdot = _d(x) @ _d(w).t() + _d(b), _d(x).abs() @ _d(w).abs().t() + _d(b).abs()
    want = hk.act(pre, slope)
    hk.faithful_bf16(got, want, absdot, f"pointwise slope={slope} faithful", max_frac=_MAX_DIFF_FRAC,
                     ulps=hk.ulps(want))


@pytest.mark.parametrize("B,h,w", [(1, 8, 16), (2, 5, 7), (1, 19, 33)])
@pytest.mark.parametrize("block", [False, True])
def test_deconv_layer(B, h, w, block):
    g = torch.Generator().manual_seed(B * 100 + h * 10 + w)
    x = _bf(torch.randn((B, h, w, 32), generator=g))
    wt = _bf(torch.randn((32, 32, 8, 8), generator=g) / 16).float()
    b = torch.randn(32, generator=g) * 0.1
    got = hk.deconv(x.to(DEV), wt, b, 0.25, block_layout=block)
    want = F.prelu(F.conv_transpose2d(x.float().permute(0, 3, 1, 2), wt, b, stride=4, padding=2),
                   torch.tensor([0.25])).permute(0, 2, 3, 1)
    if block:
        raw = got.float().cpu()
        ring = hk.to_block(torch.ones((B, 4 * h, 4 * w, 32)))      # 1 inside the image, 0 on the ring
        assert torch.isfinite(raw).all()
        assert (raw * (1 - ring)).abs().max() == 0, "padding ring of the block layout must be zero"
        got = hk.from_block(got.cpu())
    _close(got, want, f"deconv B={B} {h}x{w} block={block}")
    xc = _d(x).permute(0, 3, 1, 2)
    pre = F.conv_transpose2d(xc, _d(wt), _d(b), stride=4, padding=2).permute(0, 2, 3, 1)
    absdot = F.conv_transpose2d(xc.abs(), _d(wt).abs(), _d(b).abs(), stride=4, padding=2).permute(0, 2, 3, 1)
    want = hk.act(pre, 0.25)
    hk.faithful_bf16(got, want, absdot, f"deconv B={B} {h}x{w} block={block} faithful", max_frac=_MAX_DIFF_FRAC,
                     ulps=hk.ulps(want))


@pytest.mark.parametrize("nsrc,B,h,w", [(1, 1, 8, 16), (2, 2, 5, 7), (3, 1, 19, 33), (6, 1, 9, 17)])
def test_fused_downtran_downconv(nsrc, B, h, w):
    """The kernel the plan runs for the HR half of a feedback group (SRProjectionModule.py:70-80)."""
    g = torch.Generator().manual_seed(nsrc * 1000 + h * 10 + w)
    hr = _bf(torch.randn((nsrc, B, 4 * h, 4 * w, 32), generator=g))
    wd = _bf(torch.randn((32, 32, 8, 8), generator=g) / 45).float()
    bd = torch.randn(32, generator=g) * 0.1
    wt = _bf(torch.randn((32, 32 * nsrc), generator=g) / math.sqrt(32 * nsrc)).float()
    bt = torch.randn(32, generator=g) * 0.1
    hrb = torch.stack([hk.to_block(hr[j]) for j in range(nsrc)])
    got = hk.fused_down(hrb.to(DEV), wt, bt, 0.3, wd, bd, 0.15)
    want = _down_reference([hr[j].float() for j in range(nsrc)], wt, bt, 0.3, wd, bd, 0.15)
    _close(got, want, f"fused_down nsrc={nsrc} B={B} {h}x{w}")
    want, absdot, extra = hk.down_faithful([(_d(hr[j]), None) for j in range(nsrc)], wt, bt, 0.3, wd, bd, 0.15)
    hk.faithful_bf16(got, want, absdot, f"fused_down nsrc={nsrc} B={B} {h}x{w} faithful", max_frac=_MAX_DIFF_FRAC_FUSED,
                     extra=extra)


def _down_reference(srcs, wt, bt, slope_t, wd, bd, slope_d):
    """fp32 HR half of a feedback group: srcs = nsrc maps (B,4h,4w,32) -> cat along channels -> 1x1 (nsrc > 1) ->
    PReLU -> BF16 (the kernel rounds H to BF16 on chip) -> Conv2d(32,32,8,4,2) -> PReLU -> (B,h,w,32)."""
    x = torch.cat([s.permute(0, 3, 1, 2) for s in srcs], dim=1)
    if len(srcs) > 1:
        x = F.prelu(F.conv2d(x, wt.view(32, 32 * len(srcs), 1, 1), bt), torch.tensor([slope_t]))
        x = _bf(x).float()
    return F.prelu(F.conv2d(x, wd, bd, stride=4, padding=2), torch.tensor([slope_d])).permute(0, 2, 3, 1)


def _group_operands(nsrc, B, h, w, seed):
    """Seeded, signed, O(1) operands of one feedback group: the transposed conv's LR input, the earlier HR sources
    (plain NHWC), and the three layers' weights (rounded to BF16, as the kernels see them) and biases."""
    g = torch.Generator().manual_seed(seed)
    lr = _bf(torch.randn((B, h, w, 32), generator=g))
    prev = _bf(torch.randn((nsrc - 1, B, 4 * h, 4 * w, 32), generator=g))
    wu = _bf(torch.randn((32, 32, 8, 8), generator=g) / 16).float()
    bu = torch.randn(32, generator=g) * 0.1
    wt = _bf(torch.randn((32, 32 * nsrc), generator=g) / math.sqrt(32 * nsrc)).float()
    bt = torch.randn(32, generator=g) * 0.1
    wd = _bf(torch.randn((32, 32, 8, 8), generator=g) / 45).float()
    bd = torch.randn(32, generator=g) * 0.1
    return lr, prev, (wu, bu), (wt, bt), (wd, bd)


def _check_fused_updown(nsrc, store, B, h, w, slope_u, seed):
    """The merged kernel (transposed conv inside the down kernel) against the layered pair it replaces -- the
    standalone transposed conv into slot nsrc-1, then the fused down kernel over all nsrc slots -- bit for bit, and the
    whole group against an fp32 reference."""
    slope_t, slope_d = 0.3, 0.15
    lr, prev, (wu, bu), (wt, bt), (wd, bd) = _group_operands(nsrc, B, h, w, seed)
    lr_d = lr.to(DEV)
    u_blk = hk.deconv(lr_d, wu, bu, slope_u, block_layout=True)                       # (B,8,h+1,w+1,64)
    hr = torch.stack([hk.to_block(prev[j]).to(DEV) for j in range(nsrc - 1)] + [u_blk])
    want_y = hk.fused_down(hr, wt, bt, slope_t, wd, bd, slope_d)
    where = f"nsrc={nsrc} store={store} B={B} {h}x{w} slope_u={slope_u}"
    assert torch.isfinite(u_blk.float()).all() and torch.isfinite(want_y.float()).all(), where

    y, hr_after = hk.fused_updown(lr_d, hr, store, wu, bu, slope_u, wt, bt, slope_t, wd, bd, slope_d)
    # y of the merged kernel is the layered pair's, bit for bit (LR tile: 16 x 8 blocks -> tile (x // 16, y // 8))
    hk.bits_equal(y, want_y, f"fused_updown y vs layered pair, {where}")
    if store:   # the stored hr map is the standalone transposed conv's, zero ring included
        hk.bits_equal(hr_after[nsrc - 1], u_blk, f"fused_updown hr[{nsrc - 1}] vs transposed conv, {where}",
                      dims="b,pair,Yb,Xb,el")
    else:       # the merged kernel keeps U on chip and leaves the slot alone
        assert bool((hr_after[nsrc - 1].view(torch.int16) == hk.SENTINEL_BITS).all()), \
            f"fused_updown wrote hr[{nsrc - 1}] with store=0, {where}"
    # the two paths share packing and conventions: the whole group against fp32 as well
    u = F.prelu(F.conv_transpose2d(lr.float().permute(0, 3, 1, 2), wu, bu, stride=4, padding=2),
                torch.tensor([slope_u]))
    u = _bf(u).float().permute(0, 2, 3, 1)                   # the kernel rounds U to BF16 (it is an HR map)
    want = _down_reference([prev[j].float() for j in range(nsrc - 1)] + [u], wt, bt, slope_t, wd, bd, slope_d)
    _close(y, want, f"fused_updown vs fp32, {where}")
    lc = _d(lr).permute(0, 3, 1, 2)
    pre_u = F.conv_transpose2d(lc, _d(wu), _d(bu), stride=4, padding=2).permute(0, 2, 3, 1)
    abs_u = F.conv_transpose2d(lc.abs(), _d(wu).abs(), _d(bu).abs(), stride=4, padding=2).permute(0, 2, 3, 1)
    want, absdot, extra = hk.down_faithful([(_d(prev[j]), None) for j in range(nsrc - 1)]
                                           + [(hk.act(pre_u, slope_u), abs_u)], wt, bt, slope_t, wd, bd, slope_d)
    hk.faithful_bf16(y, want, absdot, f"fused_updown faithful, {where}", max_frac=_MAX_DIFF_FRAC_FUSED,
                     extra=extra)


# (1,7,15): exactly one 16 x 8-block tile; (1,8,16): ring blocks alone in a second tile row and column; (1,7,2370):
# 149 tiles on 148 CTAs, so one CTA walks two; (4,70,150) / (2,135,240): 360 / 544 tiles, several per CTA (the next
# tile's LR boxes are loaded while the current one runs, one D_B buffer, mbarrier parity over many tiles)
_UPDOWN_SHAPES = [(1, 1, 1), (1, 7, 15), (1, 8, 16), (2, 5, 7), (1, 19, 33), (3, 40, 61), (1, 7, 2370), (4, 70, 150),
                  (2, 135, 240)]
_UPDOWN_CASES = (
    [(n, 1) + s for n in (4, 6) for s in _UPDOWN_SHAPES]                               # the plan's nsrc: every shape
    + [(n, 1) + s for n in (2, 3, 5) for s in [(1, 8, 16), (2, 5, 7), (1, 19, 33), (3, 40, 61)]]
    + [(5, 1, 4, 70, 150), (2, 1, 1, 7, 2370), (3, 1, 1, 1, 1)]
    # store = 0: the plan's last group (hr[5] is read by no one); no TMA stores, no wait for them to read U
    + [(6, 0) + s for s in [(1, 1, 1), (1, 7, 15), (1, 19, 33), (1, 7, 2370), (4, 70, 150)]]
    + [(3, 0) + s for s in [(2, 5, 7), (3, 40, 61)]])


@pytest.mark.parametrize("nsrc,store,B,h,w", _UPDOWN_CASES)
def test_fused_updown_against_layered_pair(nsrc, store, B, h, w):
    """fused_updown_kernel (feedback groups 3-5 of the x4 stack; it accepts nsrc 2..6) at tile, ring and multi-tile
    edges: y and the stored hr map bit-identical to the layered pair, y within BF16 tolerance of fp32, guard bands
    around y and the hr array untouched, the workspace poisoned with NaN bytes."""
    _check_fused_updown(nsrc, store, B, h, w, 0.25, seed=nsrc * 7919 + B * 1000 + h * 37 + w)


@pytest.mark.parametrize("slope_u", [0.0, 1.0, -0.3, 1.7])
def test_fused_updown_prelu_slope_forms(slope_u):
    """The merged kernel's conversion of the transposed conv picks the packed-BF16 PReLU form by the slope."""
    _check_fused_updown(5, 1, 2, 19, 33, slope_u, seed=77)


@pytest.mark.parametrize("B,h,w", [(1, 8, 16), (2, 5, 7), (1, 19, 33), (1, 9, 14), (1, 17, 29), (3, 40, 61)])
def test_x2_transposed_conv_layer(B, h, w):
    """ConvTranspose2d k6 s2 p2 (x2 geometry, SURVEY.md 8 a6): staged TMA stores, ragged tiles on both axes."""
    g = torch.Generator().manual_seed(B * 100 + h * 10 + w)
    x = _bf(torch.randn((B, h, w, 32), generator=g))
    wt = _bf(torch.randn((32, 32, 6, 6), generator=g) / 12).float()
    b = torch.randn(32, generator=g) * 0.1
    got = hk.x2_layer(x.to(DEV), wt, b, 0.25, up=True)
    want = F.prelu(F.conv_transpose2d(x.float().permute(0, 3, 1, 2), wt, b, stride=2, padding=2),
                   torch.tensor([0.25])).permute(0, 2, 3, 1)
    _close(got, want, f"deconv2 B={B} {h}x{w}")
    xc = _d(x).permute(0, 3, 1, 2)
    pre = F.conv_transpose2d(xc, _d(wt), _d(b), stride=2, padding=2).permute(0, 2, 3, 1)
    absdot = F.conv_transpose2d(xc.abs(), _d(wt).abs(), _d(b).abs(), stride=2, padding=2).permute(0, 2, 3, 1)
    want = hk.act(pre, 0.25)
    hk.faithful_bf16(got, want, absdot, f"deconv2 B={B} {h}x{w} faithful", max_frac=_MAX_DIFF_FRAC,
                     ulps=hk.ulps(want))


@pytest.mark.parametrize("B,h,w", [(1, 8, 16), (2, 5, 7), (1, 19, 33), (1, 9, 14), (1, 9, 15), (1, 17, 28), (1, 17, 29),
                                   (3, 40, 61)])
def test_x2_strided_conv_layer(B, h, w):
    """Conv2d k6 s2 p2 with the column taps in output-shift form (16-column tiles finish 14): widths on both
    sides of the 14-column tile stride, zero padding through TMA fill at every border."""
    g = torch.Generator().manual_seed(B * 100 + h * 10 + w + 1)
    x = _bf(torch.randn((B, 2 * h, 2 * w, 32), generator=g))
    wd = _bf(torch.randn((32, 32, 6, 6), generator=g) / 34).float()
    b = torch.randn(32, generator=g) * 0.1
    got = hk.x2_layer(x.to(DEV), wd, b, 0.15, up=False)
    want = F.prelu(F.conv2d(x.float().permute(0, 3, 1, 2), wd, b, stride=2, padding=2),
                   torch.tensor([0.15])).permute(0, 2, 3, 1)
    _close(got, want, f"downconv2 B={B} {h}x{w}")
    xc = _d(x).permute(0, 3, 1, 2)
    pre = F.conv2d(xc, _d(wd), _d(b), stride=2, padding=2).permute(0, 2, 3, 1)
    absdot = F.conv2d(xc.abs(), _d(wd).abs(), _d(b).abs(), stride=2, padding=2).permute(0, 2, 3, 1)
    want = hk.act(pre, 0.15)
    hk.faithful_bf16(got, want, absdot, f"downconv2 B={B} {h}x{w} faithful", max_frac=_MAX_DIFF_FRAC,
                     ulps=hk.ulps(want))


def _psnr(a, b):
    mse = ((a - b) ** 2).mean().item()
    return 10 * math.log10(255.0 ** 2 / max(mse, 1e-20))


@pytest.mark.parametrize("M,h,w,steps,scale", [(8, 16, 16, 3, 4), (3, 9, 21, 2, 4), (20, 24, 40, 3, 4),
                                                (8, 16, 16, 3, 2), (3, 9, 21, 2, 2), (14, 24, 40, 3, 2), (2, 37, 19, 1, 2)])
def test_full_stack_against_oracle(M, h, w, steps, scale):
    """x4 = the reference's geometry (k8 s4 p2); x2 = SRFBN's k6 s2 p2 (BASELINE config C4; layered kernels)."""
    sd = so.init_state_dict(num_maps=M, seed=M + h, gain=2.3, upscale=scale)
    # make every slope distinct so a mixed-up layer shows
    gs = torch.Generator().manual_seed(99)
    for k in sd:
        if k.endswith(".1.weight"):
            sd[k] = torch.rand(1, generator=gs) * 0.4 + 0.05
    mod = SRProjectionModule(num_steps=steps, num_maps=M, upscale_factor=scale)
    mod.load_state_dict(sd)
    x = torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(5)) * 255
    with torch.no_grad():
        want_maps = so.forward_maps(x, sd, num_steps=steps, upscale=scale)
        # the parity test must not be blind: the conv branch (not only the bilinear skip) carries signal
        skip = F.interpolate(x, scale_factor=scale, mode="bilinear", align_corners=False)
        assert (want_maps - skip).abs().mean().item() > 0.05
        want = so.fc_fuse(want_maps, sd)
    got_maps = mod.premix(x.to(DEV)).cpu()
    got = mod(x.to(DEV)).cpu()
    assert torch.isfinite(got_maps).all() and torch.isfinite(got).all()
    # direct agreement of the per-map SR images (0..255 scale)
    assert _psnr(got_maps, want_maps) > 50.0, f"per-map PSNR {_psnr(got_maps, want_maps):.2f} dB"
    # north-star criterion: PSNR delta <= 0.05 dB against a common target ~35 dB away
    noise = torch.randn(want_maps.shape, generator=torch.Generator().manual_seed(6)) * 4.5
    target = want_maps + noise
    delta = abs(_psnr(got_maps, target) - _psnr(want_maps, target))
    assert delta <= 0.05, f"PSNR delta {delta:.4f} dB"
    # fused output: the fc mixes M maps with random weights; compare relative to its scale
    scale = want.abs().mean().item() + 1.0
    assert (got - want).abs().max().item() <= 0.02 * scale + 0.05 * (got - want).abs().mean().item() + 0.5, \
        f"fused max err {(got - want).abs().max():.4f} at scale {scale:.2f}"


@pytest.mark.parametrize("scale", [4, 2])
def test_workspace_cap_chunks_the_maps_bit_identically(scale):
    """vsr_srfbn_plan_set_workspace_cap: the plan sweeps its layers over chunks of maps (the largest divisor of M that
    fits); the maps are independent until the fc fuse, so every chunking gives the unchunked result bit for bit."""
    M, h, w = 6, 17, 26
    sd = so.init_state_dict(num_maps=M, seed=5, gain=2.3, upscale=scale)
    x = (torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(6)) * 255).to(DEV)
    ref = SRProjectionModule(num_maps=M, upscale_factor=scale)
    ref.load_state_dict(sd)
    want_maps, want = ref.premix(x), ref(x)
    ent = next(iter(ref._plans.values()))
    full = ent["workspace"].numel()
    assert ent["chunk_maps"] == M
    for frac, chunk in ((0.75, 3), (0.45, 2), (0.22, 1)):
        mod = SRProjectionModule(num_maps=M, upscale_factor=scale, workspace_cap_bytes=int(full * frac))
        mod.load_state_dict(sd)
        y = mod(x)
        e = next(iter(mod._plans.values()))
        assert e["chunk_maps"] == chunk and e["workspace"].numel() <= full * frac, (frac, e["chunk_maps"])
        assert torch.equal(y, want) and torch.equal(mod.premix(x), want_maps)
        mod.profile(True)                                   # the per-launch accounting covers every chunk sweep
        mod(x)
        prof = mod.profile_read()
        mod.profile(False)
        assert prof["im2col"]["launches"] == M // chunk and prof["fc_fuse"]["launches"] == 1
    with pytest.raises(Exception, match="workspace"):
        SRProjectionModule(num_maps=M, upscale_factor=scale, workspace_cap_bytes=1 << 16)(x)


@pytest.mark.parametrize("scale", [4, 2])
def test_plan_reads_only_workspace_bytes_written_in_the_same_forward(scale):
    """The plan's workspace may hold anything when a forward starts: the hr rings, the fp32 partial slots of the fused
    down kernels and the x4 plan's omission of hr[5] all rely on every byte a forward reads having been written by that
    forward.  A workspace filled with 0xFF bytes (NaN in BF16 and fp32) before the forward -- unchunked and chunked,
    before the first forward and again between two -- gives the frame and the per-map images of a zero-filled one,
    bit for bit."""
    M, h, w = 6, 17, 26
    sd = so.init_state_dict(num_maps=M, seed=8, gain=2.3, upscale=scale)
    x = (torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(9)) * 255).to(DEV)

    def module(poison, cap=None):
        mod = SRProjectionModule(num_maps=M, upscale_factor=scale, workspace_cap_bytes=cap)
        mod.load_state_dict(sd)
        ent = mod._plan_for(M, h, w, x.device)
        ent["workspace"].fill_(0xFF if poison else 0)
        return mod, ent

    clean, ent = module(False)
    want, want_maps = clean(x), clean.premix(x)
    assert torch.isfinite(want).all() and torch.isfinite(want_maps).all()
    full = ent["workspace"].numel()
    for cap in (None, int(full * 0.45)):
        mod, ent = module(True, cap)
        assert ent["chunk_maps"] == (M if cap is None else 2)
        assert torch.equal(mod(x).view(torch.int32), want.view(torch.int32)), cap
        ent["workspace"].fill_(0xFF)                     # poisoned again between two full forwards
        got_maps = mod.premix(x)
        assert torch.equal(got_maps.view(torch.int32), want_maps.view(torch.int32)), cap
        ent["workspace"].fill_(0xFF)
        assert torch.equal(mod(x).view(torch.int32), want.view(torch.int32)), cap
        del mod


@pytest.mark.parametrize("scale", [4, 2])
def test_refresh_of_the_changed_maps_is_bit_identical_to_a_full_forward(scale):
    """forward(x, changed_from=k): only the maps x[k:] go through the conv stack again, the per-map images of x[:k]
    come from the previous forward (the maps are independent until the fc fuse) -- the frame and the per-map images
    equal a full forward's bit for bit, for every k, repeatedly, and the call refuses to run without a preceding full
    forward or on a chunked plan."""
    M, h, w = 8, 19, 27
    sd = so.init_state_dict(num_maps=M, seed=3, gain=2.3, upscale=scale)
    g = torch.Generator().manual_seed(11)
    x = (torch.rand((M, 3, h, w), generator=g) * 255).to(DEV)
    ref = SRProjectionModule(num_maps=M, upscale_factor=scale)
    ref.load_state_dict(sd)
    mod = SRProjectionModule(num_maps=M, upscale_factor=scale)
    mod.load_state_dict(sd)
    with pytest.raises(RuntimeError, match="preceding full forward"):
        mod(x, changed_from=3)
    for k in (3, M - 1, 1, 3):
        x2 = x.clone()
        x2[k:] = (torch.rand((M - k, 3, h, w), generator=g) * 255).to(DEV)
        want, want_maps = ref(x2), ref.premix(x2)
        mod(x)                                               # pass 1 on the old stack
        u8 = torch.zeros((scale * h, scale * w, 3), dtype=torch.uint8, device=DEV)
        got = mod(x2, out_u8=u8, changed_from=k)             # pass 2: maps k.. changed
        assert torch.equal(got, want), k
        ent = next(iter(mod._plans.values()))
        maps = torch.empty_like(want_maps)
        from video_super_resolution_b200 import _lib
        _lib.check(_lib.lib().vsr_srfbn_debug_premix(ent["plan"], maps.data_ptr(), torch.cuda.current_stream().cuda_stream), "premix")
        assert torch.equal(maps, want_maps), k
        got2 = mod(x2, changed_from=k)                       # again on top of a refreshed premix buffer: still exact
        assert torch.equal(got2, want), k
    capped = SRProjectionModule(num_maps=M, upscale_factor=scale,
                                workspace_cap_bytes=next(iter(ref._plans.values()))["workspace"].numel() // 2)
    capped.load_state_dict(sd)
    capped(x)
    with pytest.raises(RuntimeError, match="srfbn_prepare_refresh"):
        capped(x, changed_from=3)
