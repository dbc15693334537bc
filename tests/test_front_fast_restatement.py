"""The CPU restatement of the front's fast arithmetic (oracle.or_warp_nhwc_fast, oracle.or_compose_flow_fast): the mode-2
warp and the flow chain that WarpFusePipeline runs.  No GPU: these check the restatement itself, so that the GPU tests
that hold the kernels to it bit for bit (test_front_faithful_gpu) pin the right arithmetic.

An independent numpy restatement (`_blend_np`, fp32 products and a correctly rounded fmaf built from fp64) must give the
C restatement's bits; the same numpy code with the operands of one FMA swapped, or with the FMAs split into a product
and a sum, must not."""
import numpy as np
import pytest

from oracle import oracle as orc
from video_super_resolution_b200 import synthetic

F32, F64 = np.float32, np.float64


def _fmaf(a, b, c):
    """Correctly rounded fp32 fma(a, b, c) for finite fp32 arrays: the product is exact in fp64; the fp64 sum's rounding
    error (TwoSum) decides the one case where rounding fp64 -> fp32 would round twice (an fp64 sum on an fp32 midpoint)."""
    a, b, c = (np.asarray(v, F32) for v in (a, b, c))
    p = a.astype(F64) * b.astype(F64)
    c64 = c.astype(F64)
    s = p + c64
    bb = s - p
    e = (p - (s - bb)) + (c64 - bb)              # s + e == p + c exactly
    r = s.astype(F32)
    r64 = r.astype(F64)
    other = np.nextafter(r, np.where(s > r64, F32(np.inf), F32(-np.inf)))
    mid = (s != r64) & ((r64 + other.astype(F64)) * 0.5 == s)
    fix = mid & (np.sign(e) == np.sign(other.astype(F64) - r64))
    return np.where(fix, other, r).astype(F32)


def _taps(flow, H, W):
    """Tap indices (flattened y*W+x) and fp32 fractions of the fast warp, for an (H,W,2) flow."""
    yy, xx = np.meshgrid(np.arange(H, dtype=F32), np.arange(W, dtype=F32), indexing="ij")
    xf = (xx + flow[..., 0]).astype(F32)
    yf = (yy + flow[..., 1]).astype(F32)
    fx0, fy0 = np.floor(xf), np.floor(yf)
    xL = np.clip(fx0, 0, W - 1).astype(np.int64)
    xR = np.clip(fx0 + F32(1), 0, W - 1).astype(np.int64)
    yT = np.clip(fy0, 0, H - 1).astype(np.int64)
    yB = np.clip(fy0 + F32(1), 0, H - 1).astype(np.int64)
    return (yT * W + xL, yT * W + xR, yB * W + xL, yB * W + xR), (xf - fx0).astype(F32), (yf - fy0).astype(F32)


def _blend_np(src, flow, variant="faithful"):
    """numpy restatement of the fast warp of one (H,W,C) image.  variant: "faithful" (blend_fast of warp.cu),
    "swap_top" (top = fma(ia, tl, a*tr)), "swap_rows" (v = fma(ib, top, b*bot)), "unfused" (every fma a product and a
    sum, each rounded)."""
    H, W, C = src.shape
    (tl, tr, bl, br), a, b = _taps(flow, H, W)
    s = src.reshape(H * W, C)
    TL, TR, BL, BR = (s[i.ravel()].reshape(H, W, C) for i in (tl, tr, bl, br))
    a, b = a[..., None], b[..., None]
    ia, ib = (F32(1) - a).astype(F32), (F32(1) - b).astype(F32)
    fma = _fmaf if variant != "unfused" else (lambda x, y, z: (x * y).astype(F32) + z)
    if variant == "swap_top":
        top = fma(ia, TL, (a * TR).astype(F32))
    else:
        top = fma(a, TR, (ia * TL).astype(F32))
    bot = fma(a, BR, (ia * BL).astype(F32))
    if variant == "swap_rows":
        return fma(ib, top, (b * bot).astype(F32))
    return fma(b, bot, (ib * top).astype(F32))


def _case(seed, B=2, H=23, W=41, C=3, mag=6.0):
    rng = np.random.default_rng(seed)
    src = (rng.random((B, H, W, C)) * 255).astype(F32)
    flow = synthetic.smooth_flow(B, H, W, mag, seed=seed).numpy() + (rng.random((B, H, W, 2)) - 0.5).astype(F32)
    return src, flow.astype(F32)


@pytest.mark.parametrize("C", [1, 3, 5, 8])
def test_fast_mode_is_a_faithful_bilinear_and_not_the_exact_mode(C):
    src, flow = _case(C, C=C)
    fast = orc.warp_nhwc(src, flow, 2)
    exact = orc.warp_nhwc(src, flow, True)
    B, H, W, _ = src.shape
    for bi in range(B):
        (tl, tr, bl, br), a, b = _taps(flow[bi], H, W)
        s = src[bi].reshape(H * W, C).astype(F64)
        a, b = a[..., None].astype(F64), b[..., None].astype(F64)
        TL, TR, BL, BR = (s[i.ravel()].reshape(H, W, C) for i in (tl, tr, bl, br))
        want = (1 - b) * ((1 - a) * TL + a * TR) + b * ((1 - a) * BL + a * BR)      # plain fp64 bilinear, same taps
        big = np.maximum.reduce([np.abs(TL), np.abs(TR), np.abs(BL), np.abs(BR)]).astype(F32)
        ulp = np.spacing(big).astype(F64)
        # fp32 ia*tl, two FMAs per row and one across: about 3 roundings of values <= the largest tap
        assert (np.abs(fast[bi] - want) <= 3 * ulp).all(), np.abs(fast[bi] - want).max()
    assert np.abs(fast - exact).max() <= 1e-4
    assert not np.array_equal(fast, exact)                 # the fast mode, not the exact one under another name


def test_fast_mode_matches_an_independent_restatement_and_catches_reorderings():
    src, flow = _case(11, B=1, H=31, W=47, C=3)
    fast = orc.warp_nhwc(src, flow, 2)[0]
    assert np.array_equal(fast, _blend_np(src[0], flow[0]))
    for variant in ("swap_top", "swap_rows", "unfused"):
        assert not np.array_equal(fast, _blend_np(src[0], flow[0], variant)), variant


def test_fused_residual_is_the_channel_norm_of_the_fast_warp():
    src, flow = _case(12, C=3)
    ref = (np.random.default_rng(3).random(src.shape) * 255).astype(F32)
    warped, norm = orc.warp_nhwc(src, flow, 2, ref=ref)
    assert np.array_equal(warped, orc.warp_nhwc(src, flow, 2))
    assert np.array_equal(norm, orc.channelnorm_nhwc(ref - warped))   # fp32 difference, fmaf chain, sqrtf


def test_integer_flows_return_the_source_bits():
    B, H, W, C = 1, 17, 29, 3
    rng = np.random.default_rng(5)
    src = (rng.random((B, H, W, C)) * 255).astype(F32)
    flow = rng.integers(-3, 4, (B, H, W, 2)).astype(F32)
    got = orc.warp_nhwc(src, flow, 2)
    yy, xx = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    ys = np.clip(yy + flow[0, ..., 1].astype(int), 0, H - 1)
    xs = np.clip(xx + flow[0, ..., 0].astype(int), 0, W - 1)
    assert np.array_equal(got[0].view(np.uint32), src[0, ys, xs].view(np.uint32))
    f = synthetic.smooth_flow(1, H, W, 5.0, seed=2).numpy()[0]
    assert np.array_equal(orc.compose_flow(None, f, fast=True), f)      # the identity link of the chain


def test_compose_flow_fast_is_g_plus_the_fast_warp_of_f():
    g = synthetic.smooth_flow(1, 40, 56, 6.0, seed=1).numpy()[0]
    f = synthetic.smooth_flow(1, 40, 56, 6.0, seed=2).numpy()[0]
    got = orc.compose_flow(g, f, fast=True, threads=3)
    assert np.array_equal(got, (g + orc.warp_nhwc(f[None], g[None], 2)[0]).astype(F32))
    assert np.array_equal(got, (g + _blend_np(f, g)).astype(F32))
    exact = orc.compose_flow(g, f)
    assert 0 < np.abs(got - exact).max() <= 1e-5


def test_pinned_case_where_the_fma_is_fused():
    """Found by a seeded search: a 2x2 image sampled at (a, b) from pixel (0, 0), where the fused blend and the same
    sequence with every product rounded on its own (and the exact mode) give different fp32 bits."""
    a, b = np.array([1062671694, 1038497019], np.uint32).view(F32)
    taps = np.array([1125775026, 1123312613, 1125623047, 1126702457], np.uint32).view(F32)   # tl, tr, bl, br
    src = taps.reshape(1, 2, 2, 1)
    flow = np.zeros((1, 2, 2, 2), F32)
    flow[0, 0, 0] = (a, b)
    got = orc.warp_nhwc(src, flow, 2)[0, 0, 0, 0]
    assert got.view(np.uint32) == 1124307287
    assert _blend_np(src[0], flow[0], "unfused")[0, 0, 0].view(np.uint32) == 1124307286
    assert orc.warp_nhwc(src, flow, True)[0, 0, 0, 0].view(np.uint32) == 1124307286


def test_huge_and_nan_flows_follow_the_exact_modes_taps():
    src, flow = _case(21, B=1, H=9, W=33, C=3)
    flow[0, 1, 1] = (5e6, -5e6)
    flow[0, 2, 2] = (-3e38, 3e38)
    flow[0, 3, 3] = (np.nan, 1.0)
    flow[0, 4, 4] = (-4194304.5, 4194303.5)
    fast = orc.warp_nhwc(src, flow, 2)
    exact = orc.warp_nhwc(src, flow, True)
    for y, x in ((1, 1), (2, 2), (4, 4)):        # integral coordinates: both modes return the clamped tap's bits
        assert np.array_equal(fast[0, y, x], exact[0, y, x]), (y, x)
    assert np.isnan(fast[0, 3, 3]).all() == np.isnan(exact[0, 3, 3]).all()


def test_chain_and_front_restatement_keep_the_exact_callers():
    """fast=False keeps what the exact restatement returned before it had a fast mode; fast=True runs the
    restated chain and warp, and W windows are one restatement per window."""
    T, h, w = 5, 20, 28
    fr = synthetic.frames(T, h, w, seed=1).numpy()
    fl = synthetic.smooth_flow(T - 1, h, w, 4.0, seed=2).numpy()
    d = synthetic.inv_depth(T - 1, h, w, seed=3).numpy()
    la, lb = (x.numpy() for x in synthetic.logits(h, w, seed=4))
    stack, r = orc.warp_fuse_front(fr, fl, d, la, lb)
    c = T // 2
    proj_d = orc.flow_projection(fl, d)[0]
    G = orc.chain_flows(proj_d, fl, c)
    assert np.array_equal(G[c - 1], proj_d[c - 1]) and np.array_equal(G[c], fl[c])
    assert np.array_equal(G[c - 2], orc.compose_flow(G[c - 1], proj_d[c - 2]))
    assert np.array_equal(r["centre_flows"], G)
    neigh = fr[[t for t in range(T) if t != c]]
    assert np.array_equal(r["warped"], orc.warp_nhwc(neigh, G, True))
    assert np.array_equal(r["resid"], orc.channelnorm_nhwc(fr[c][None] - r["warped"]))
    stack_f, rf = orc.warp_fuse_front(fr, fl, d, la, lb, fast=True, threads=2)
    Gf = orc.chain_flows(proj_d, fl, c, fast=True)
    assert np.array_equal(rf["centre_flows"], Gf)
    assert np.array_equal(rf["warped"], orc.warp_nhwc(neigh, Gf, 2))
    assert 0 < np.abs(stack_f - stack).max() <= 1e-2
    # W = 2 windows: window 1 is another seed
    fr2, fl2, d2 = synthetic.frames(T, h, w, seed=5).numpy(), synthetic.smooth_flow(T - 1, h, w, 4.0, seed=6).numpy(), d[::-1].copy()
    sW, rW = orc.warp_fuse_front(np.stack([fr, fr2]), np.stack([fl, fl2]), np.stack([d, d2]), np.stack([la, lb]),
                                 np.stack([lb, la]), fast=True)
    s2, r2 = orc.warp_fuse_front(fr2, fl2, d2, lb, la, fast=True)
    assert np.array_equal(sW[0], stack_f) and np.array_equal(sW[1], s2)
    assert all(np.array_equal(rW[k][1], r2[k]) for k in r2)
    # given projections replace the restated ones; everything downstream follows them
    nudged = (rf["proj_depth"] + F32(0.25)).astype(F32)
    _, rp = orc.warp_fuse_front(fr, fl, d, la, lb, fast=True, projected=(rf["proj_flow"], nudged, rf["wsum"]))
    assert np.array_equal(rp["centre_flows"], orc.chain_flows(nudged, fl, c, fast=True))
