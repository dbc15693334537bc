"""Python front-ends of the single-layer test hooks of the C ABI (vsr_test_*), the plan walk hooks
(vsr_srfbn_debug_run_layers / vsr_srfbn_debug_buffer), the HR block layout helpers, the float64 expectations the
layer tests share, and the full-size cases, state dict and per-region error measures of the whole-stack tests.  Test
support only."""
import ctypes

import torch
import torch.nn.functional as F

from oracle import srfbn_bf16 as sb
from oracle import srfbn_oracle as so
from video_super_resolution_b200 import _lib

# activation buffer ids of vsr_srfbn_debug_buffer (include/vsr_b200.h VSR_SRFBN_BUF_*)
BUF_A0, BUF_C128, BUF_XFEAT, BUF_HIDDEN, BUF_LR, BUF_U, BUF_HR, BUF_HB, BUF_HT, BUF_ACC, BUF_PREMIX = range(11)

# The full-size plans of test_srfbn_faithful_gpu.py::test_full_size_maps_against_restatement and
# test_fullsize_gpu.py::test_full_size_windows_bit_identical: name -> (M, h, w, scale, windows, workspace cap in bytes or
# None).  tests/test_srfbn_plan_buffers_cpu.py checks that each still reaches the size it exists for.
FULL_SIZE_PLANS = {
    "C2": (20, 270, 480, 4, 1, None),                 # bench C2: the HR ring over 2^31 bytes
    "C5": (8, 360, 720, 4, 1, None),                  # bench C5: every map restated, so the fused frame is too
    "C4": (14, 1080, 1920, 2, 1, None),               # bench C4, uncapped: buffers over 2^31 BF16 elements
    "C5-W3": (8, 360, 720, 4, 3, None),               # 24 maps in one chunk: the HR ring over 2^32 bytes
    "C5-W3-capped": (8, 360, 720, 4, 3, 14 << 30),    # chunks of 6 maps that straddle the window boundaries
    "C2-W2": (20, 270, 480, 4, 2, None),              # 40 maps in one chunk: the HR ring over 2^32 bytes
}


def stack_state(M, h, scale):
    """The state dict of test_full_stack_against_oracle with distinct slopes, plus one layer at slope 1.3 and one at
    -0.2, so the stack runs all three packed-PReLU forms (and the fp32 PReLU of the x4 strided convs)."""
    sd = so.init_state_dict(num_maps=M, seed=M + h, gain=2.3, upscale=scale)
    gs = torch.Generator().manual_seed(99)
    for k in sd:
        if k.endswith(".1.weight"):
            sd[k] = torch.rand(1, generator=gs) * 0.4 + 0.05
    sd["block.upBlocks.2.1.weight"] = torch.tensor([1.3])
    sd["block.compress_in.1.weight"] = torch.tensor([-0.2])
    sd["fc.2.weight"] = sd["fc.2.weight"].abs()          # a fused frame the final ReLU does not zero
    return sd


def fc_fuse_bound(maps, sd):
    """Per-element error bound of the fused frame against an fp64 fc (sb.fc_fuse) over the same per-map images maps
    (M,3,H,W): twice the error bound of the kernel's fp32 FMA chains (hid_j: M + 1 terms, o: 33 terms), on the maps'
    device, (1,3,H,W) float64.  Elementwise, so it may be taken over any slice of the channels, rows or columns."""
    dev, M = maps.device, maps.shape[0]

    def d(t):
        return t.to(dev, torch.float64)

    w0, b0, w2, b2 = (d(sd[k]) for k in ("fc.0.weight", "fc.0.bias", "fc.2.weight", "fc.2.bias"))
    t = maps.double().permute(1, 2, 3, 0)
    hid = F.relu(F.linear(t, w0, b0))
    u = 2.0 ** -24
    bound = 33 * u * F.linear(hid, w2.abs(), b2.abs())
    del hid
    bound += F.linear((M + 1) * u * F.linear(t.abs(), w0.abs(), b0.abs()), w2.abs())
    return 2 * bound.permute(3, 0, 1, 2) + 1e-30


# ---- per-region errors of whole maps ------------------------------------------------------------------------------
def regions(H, W, scale):
    """The regions region_errors reports on an H x W HR map, as (name, y0, y1, x0, x1) in HR pixels: the outermost
    2 * scale HR rows and columns on each side as four bands (the (h+1) x (w+1) block ring and the ragged last tiles
    meet there), then a grid of tiles over 32 x 32 LR blocks (ragged at the bottom and right), named in LR pixels."""
    e, t = 2 * scale, 32 * scale
    out = [("top band", 0, e, 0, W), ("bottom band", H - e, H, 0, W), ("left band", 0, H, 0, e),
           ("right band", 0, H, W - e, W)]
    for y0 in range(0, H, t):
        for x0 in range(0, W, t):
            y1, x1 = min(y0 + t, H), min(x0 + t, W)
            out.append((f"tile LR y {y0 // scale}:{y1 // scale} x {x0 // scale}:{x1 // scale}", y0, y1, x0, x1))
    return out


def region_errors(got, want, scale):
    """Per-map, per-region max-abs and RMS of got - want, maps (n,3,H,W) on any devices (computed in float64 on got's):
    -> (regions(H, W, scale), max (n, R), RMS (n, R)), the two on the CPU."""
    err = got.double() - want.to(got.device, torch.float64)
    n, _, H, W = err.shape
    regs = regions(H, W, scale)
    t = 32 * scale
    ty, tx = -(-H // t), -(-W // t)
    pad = (0, tx * t - W, 0, ty * t - H)
    mx, ss, cnt = [], [], []
    for _, y0, y1, x0, x1 in regs[:4]:
        band = err[:, :, y0:y1, x0:x1]
        mx.append(band.abs().amax(dim=(1, 2, 3)))
        ss.append(band.square().sum(dim=(1, 2, 3)))
    tiles = F.pad(err, pad).view(n, 3, ty, t, tx, t)
    mx = torch.cat([torch.stack(mx, 1), tiles.abs().amax(dim=(1, 3, 5)).flatten(1)], 1)
    ss = torch.cat([torch.stack(ss, 1), tiles.square().sum(dim=(1, 3, 5)).flatten(1)], 1)
    cnt = torch.tensor([3.0 * (y1 - y0) * (x1 - x0) for _, y0, y1, x0, x1 in regs], dtype=torch.float64,
                       device=err.device)
    return regs, mx.cpu(), (ss / cnt).sqrt().cpu()


def region_failures(regs, mx, rms, b_max, b_rms, maps):
    """One line per (map, region) of region_errors whose max-abs exceeds b_max or whose RMS exceeds b_rms; maps names
    the rows of mx and rms."""
    bad = ((mx > b_max) | (rms > b_rms)).nonzero().tolist()
    return [f"map {maps[i]} {regs[r][0]}: max {mx[i, r].item():.4g} (bound {b_max}) rms {rms[i, r].item():.4g} "
            f"(bound {b_rms})" for i, r in bad]


def _fp(t):
    return ctypes.cast(t.data_ptr(), ctypes.c_void_p)


def to_block(x):
    """(B,4h,4w,C) plain NHWC -> HR block layout (B,8,h+1,w+1,2*C): blocks of 4x4 pixels whose origin is
    shifted by (-2,-2) (zero ring outside the image), stored as 8 planes of sub-position pairs
    (s = ry*4+rx, pair = s>>1): element [b, pair, Yb, Xb, (s&1)*C + c]."""
    B, H, W, C = x.shape
    xp = torch.nn.functional.pad(x, (0, 0, 2, 2, 2, 2))
    xp = xp.view(B, H // 4 + 1, 4, W // 4 + 1, 4, C)                 # b, Yb, ry, Xb, rx, c
    xp = xp.permute(0, 2, 4, 1, 3, 5)                                 # b, ry, rx, Yb, Xb, c
    xp = xp.reshape(B, 8, 2, H // 4 + 1, W // 4 + 1, C)               # b, pair, s&1, Yb, Xb, c
    return xp.permute(0, 1, 3, 4, 2, 5).reshape(B, 8, H // 4 + 1, W // 4 + 1, 2 * C).contiguous()


def from_block(xb):
    B, _, hb, wb, C2 = xb.shape
    C = C2 // 2
    x = xb.view(B, 8, hb, wb, 2, C).permute(0, 1, 4, 2, 3, 5).reshape(B, 4, 4, hb, wb, C)   # b, ry, rx, Yb, Xb, c
    x = x.permute(0, 3, 1, 4, 2, 5).reshape(B, hb * 4, wb * 4, C)
    return x[:, 2:-2, 2:-2].contiguous()


def _ws(dev):
    n = int(_lib.lib().vsr_test_workspace_bytes(1, 1, 1))
    return torch.empty(n, dtype=torch.uint8, device=dev)


def pointwise(x_bf16, w, b, slope, act=True):
    """x (rows,K) bf16 cuda; w (32,K) f32 cpu; b (32) f32 cpu -> (rows,32) bf16."""
    rows, K = x_bf16.shape
    y = torch.empty((rows, 32), dtype=torch.bfloat16, device=x_bf16.device)
    ws = _ws(x_bf16.device)
    w = w.contiguous().float()
    b = b.contiguous().float()
    _lib.check(_lib.lib().vsr_test_pointwise(x_bf16.data_ptr(), rows, K, _fp(w), _fp(b), float(slope), int(act),
                                             y.data_ptr(), ws.data_ptr(), ws.numel(),
                                             torch.cuda.current_stream().cuda_stream), "test_pointwise")
    return y


def deconv(x_bf16, w, b, slope, block_layout=False):
    """x (B,h,w,32) bf16; w (32,32,8,8) ConvTranspose layout -> (B,4h,4w,32) or block layout."""
    B, h, wd, _ = x_bf16.shape
    shape = (B, 8, h + 1, wd + 1, 64) if block_layout else (B, 4 * h, 4 * wd, 32)
    y = torch.full(shape, float("nan"), dtype=torch.bfloat16, device=x_bf16.device)
    ws = _ws(x_bf16.device)
    w = w.contiguous().float()
    b = b.contiguous().float()
    _lib.check(_lib.lib().vsr_test_deconv(x_bf16.data_ptr(), B, h, wd, _fp(w), _fp(b), float(slope),
                                          int(block_layout), y.data_ptr(), ws.data_ptr(), ws.numel(),
                                          torch.cuda.current_stream().cuda_stream), "test_deconv")
    return y


def x2_layer(x_bf16, w, b, slope, up):
    """x2 geometry (k6 s2 p2): up: x (B,h,w,32) -> (B,2h,2w,32), w (32 in,32 out,6,6); down: x (B,2h,2w,32) ->
    (B,h,w,32), w (32 out,32 in,6,6).  The output sits between two guard bands that must come back untouched
    (the kernels store through clipped TMA boxes / predicated register stores)."""
    B, H, W, _ = x_bf16.shape
    h, wd = (H, W) if up else (H // 2, W // 2)
    shape = (B, 2 * h, 2 * wd, 32) if up else (B, h, wd, 32)
    n = shape[0] * shape[1] * shape[2] * shape[3]
    G = 1 << 16                                   # guard elements on each side (128 KB: more than a tile row)
    buf = torch.full((n + 2 * G,), 12345.0, dtype=torch.bfloat16, device=x_bf16.device)
    y = buf[G:G + n].view(shape)
    y.fill_(float("nan"))
    ws = _ws(x_bf16.device)
    w = w.contiguous().float()
    b = b.contiguous().float()
    _lib.check(_lib.lib().vsr_test_x2_layer(x_bf16.data_ptr(), int(up), B, h, wd, _fp(w), _fp(b), float(slope),
                                            y.data_ptr(), ws.data_ptr(), ws.numel(),
                                            torch.cuda.current_stream().cuda_stream), "test_x2_layer")
    assert bool((buf[:G] == 12345.0).all()) and bool((buf[G + n:] == 12345.0).all()), "x2 layer wrote outside its output"
    return y.clone()


def fused_down(hr_bf16, wt, bt, slope_t, wd, bd, slope_d):
    """hr (nsrc,B,8,h+1,w+1,64) bf16 block layout; wt (32,32*nsrc)|None; wd (32,32,8,8) -> (B,h,w,32) bf16."""
    nsrc, B, _, hb, wb = hr_bf16.shape[:5]
    h, wd_ = hb - 1, wb - 1
    dev = hr_bf16.device
    y = torch.full((B, h, wd_, 32), float("nan"), dtype=torch.bfloat16, device=dev)
    n = int(_lib.lib().vsr_test_workspace_bytes(B, h, wd_)) + B * h * wd_ * 512
    ws = torch.full((n,), 0xFF, dtype=torch.uint8, device=dev)   # the fp32 partial slots start as NaN
    wd = wd.contiguous().float()
    bd = bd.contiguous().float()
    if nsrc > 1:
        wt = wt.contiguous().float()
        bt = bt.contiguous().float()
    _lib.check(_lib.lib().vsr_test_fused_down(hr_bf16.data_ptr(), nsrc, B, h, wd_,
                                              _fp(wt) if nsrc > 1 else None, _fp(bt) if nsrc > 1 else None,
                                              float(slope_t), _fp(wd), _fp(bd), float(slope_d), y.data_ptr(),
                                              ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream),
               "test_fused_down")
    return y


GUARD_BITS = 0x1234          # bf16 bit pattern of the guard bands
SENTINEL_BITS = 0x5A5A       # bf16 bit pattern of an hr slot the kernel must not write


def _guarded(shape, dev):
    """A bf16 tensor of `shape` between two guard bands of GUARD_BITS; returns (whole buffer, tensor, guard size)."""
    n = 1
    for s in shape:
        n *= s
    G = 1 << 16                                   # guard elements on each side (128 KB: more than a tile row)
    buf = torch.empty((n + 2 * G,), dtype=torch.bfloat16, device=dev)
    buf.view(torch.int16).fill_(GUARD_BITS)
    return buf, buf[G:G + n].view(shape), G


def _guards_intact(buf, G):
    bits = buf.view(torch.int16)
    return bool((bits[:G] == GUARD_BITS).all()) and bool((bits[-G:] == GUARD_BITS).all())


def fused_updown(lr_bf16, hr_bf16, store, wu, bu, slope_u, wt, bt, slope_t, wd, bd, slope_d):
    """One feedback group through the merged kernel (vsr_test_fused_updown).  lr (B,h,w,32) bf16: the transposed conv's
    input; hr (nsrc,B,8,h+1,w+1,64) bf16 block layout: slots 0..nsrc-2 are the earlier sources (slot nsrc-1 is not
    read from the caller's tensor); wu (32 in,32 out,8,8); wt (32,32*nsrc); wd (32,32,8,8).
    Returns (y (B,h,w,32), the hr array after the call).  y and the hr array sit between guard bands that must come back
    untouched; y starts as NaN, slot nsrc-1 as NaN (store) or SENTINEL_BITS (not store), the workspace (weights and fp32
    partial slots) as 0xFF bytes; slots 0..nsrc-2 must come back unchanged."""
    nsrc, B, _, hb, wb = hr_bf16.shape[:5]
    h, w_ = hb - 1, wb - 1
    dev = lr_bf16.device
    assert tuple(lr_bf16.shape) == (B, h, w_, 32)
    hbuf, hr, Gh = _guarded(tuple(hr_bf16.shape), dev)
    hr[:nsrc - 1].copy_(hr_bf16[:nsrc - 1])
    if store:
        hr[nsrc - 1].fill_(float("nan"))
    else:
        hr[nsrc - 1].view(torch.int16).fill_(SENTINEL_BITS)
    ybuf, y, Gy = _guarded((B, h, w_, 32), dev)
    y.fill_(float("nan"))
    n = int(_lib.lib().vsr_test_workspace_bytes(B, h, w_)) + B * h * w_ * 512
    ws = torch.full((n,), 0xFF, dtype=torch.uint8, device=dev)
    wu, bu, wt, bt, wd, bd = (t.contiguous().float() for t in (wu, bu, wt, bt, wd, bd))
    _lib.check(_lib.lib().vsr_test_fused_updown(lr_bf16.data_ptr(), hr.data_ptr(), nsrc, int(store), B, h, w_,
                                                _fp(wu), _fp(bu), float(slope_u), _fp(wt), _fp(bt), float(slope_t),
                                                _fp(wd), _fp(bd), float(slope_d), y.data_ptr(), ws.data_ptr(),
                                                ws.numel(), torch.cuda.current_stream().cuda_stream),
               "test_fused_updown")
    assert _guards_intact(ybuf, Gy), "fused_updown wrote outside y"
    assert _guards_intact(hbuf, Gh), "fused_updown wrote outside the hr array"
    assert torch.equal(hr[:nsrc - 1].view(torch.int16), hr_bf16[:nsrc - 1].view(torch.int16)), \
        "fused_updown wrote into a source slot it only reads"
    return y.clone(), hr.clone()


def conv_in(x, w, b, slope, sub_bias):
    """x (B,3,h,w) f32 cuda; w (128,3,3,3), b (128), sub_bias (3) f32 cpu -> (B,h,w,128) bf16 (vsr_test_conv_in).  y
    starts as NaN between two guard bands that must come back untouched; the workspace starts as 0xFF bytes."""
    B, _, h, w_ = x.shape
    ybuf, y, G = _guarded((B, h, w_, 128), x.device)
    y.fill_(float("nan"))
    n = int(_lib.lib().vsr_test_workspace_bytes(B, h, w_)) + B * h * w_ * 64
    ws = torch.full((n,), 0xFF, dtype=torch.uint8, device=x.device)
    x = x.contiguous().float()
    w, b, sub_bias = (t.contiguous().float() for t in (w, b, sub_bias))
    _lib.check(_lib.lib().vsr_test_conv_in(x.data_ptr(), B, h, w_, _fp(w), _fp(b), float(slope), _fp(sub_bias),
                                           y.data_ptr(), ws.data_ptr(), ws.numel(),
                                           torch.cuda.current_stream().cuda_stream), "test_conv_in")
    assert _guards_intact(ybuf, G), "conv_in wrote outside y"
    return y.clone()


F32_GUARD = 1234.5           # value of the fp32 guard bands around conv_out's output


def conv_out(hb_bf16, x, scale, w, b, sub_bias, add_bias):
    """hb (B,s*h,s*w,32) bf16 cuda; x (B,3,h,w) f32 cuda; w (3,32,3,3), b (3), sub_bias (3), add_bias (3) f32 cpu ->
    (B,3,s*h,s*w) f32 (vsr_test_conv_out).  y starts as NaN between two fp32 guard bands that must come back
    untouched."""
    B, _, h, w_ = x.shape
    assert tuple(hb_bf16.shape) == (B, scale * h, scale * w_, 32)
    n = B * 3 * scale * h * scale * w_
    G = 1 << 15                                   # 128 KB on each side: more than one output row of a tile
    buf = torch.full((n + 2 * G,), F32_GUARD, dtype=torch.float32, device=x.device)
    y = buf[G:G + n].view(B, 3, scale * h, scale * w_)
    y.fill_(float("nan"))
    ws = _ws(x.device)
    x = x.contiguous().float()
    w, b, sub_bias, add_bias = (t.contiguous().float() for t in (w, b, sub_bias, add_bias))
    _lib.check(_lib.lib().vsr_test_conv_out(hb_bf16.data_ptr(), x.data_ptr(), int(scale), B, h, w_, _fp(w), _fp(b),
                                            _fp(sub_bias), _fp(add_bias), y.data_ptr(), ws.data_ptr(), ws.numel(),
                                            torch.cuda.current_stream().cuda_stream), "test_conv_out")
    assert bool((buf[:G] == F32_GUARD).all()) and bool((buf[G + n:] == F32_GUARD).all()), "conv_out wrote outside y"
    return y.clone()


def faithful_bf16(got, want, absdot, what, c=16.0, max_frac=None, ulps=1, extra=0.0):
    """BF16 outputs of one layer fed the restatement's own BF16 inputs: |got - want| <= ulps * ulp_bf16(want) +
    c * 2^-24 * absdot + extra per element, absdot = sum |w * x| (the fp32 accumulation error, cancellation included);
    and the fraction of elements that differ at all <= max_frac.  ulps is 1, or 2 where a second BF16 rounding follows
    the first (the negative side of the packed PReLU: bf16(s * bf16(x)), so one ulp of x may become two of the
    output); extra covers an intermediate BF16 value that rounds the other way (see the fused down tests).  Returns
    (fraction that differs, worst err / tolerance)."""
    got, want, absdot = (t.double().cpu() for t in (got, want, absdot))
    ulps = ulps.double().cpu() if torch.is_tensor(ulps) else ulps
    extra = extra.double().cpu() if torch.is_tensor(extra) else extra
    assert torch.isfinite(got).all(), f"{what}: non-finite output"
    ulp = torch.exp2(torch.floor(torch.log2(want.abs().clamp_min(2.0 ** -126))) - 7)
    tol = ulps * ulp + c * 2.0 ** -24 * absdot + extra
    err = (got - want).abs()
    bad = (err > tol).nonzero()
    if bad.numel():
        first = [tuple(i.tolist()) for i in bad[:6]]
        raise AssertionError(f"{what}: {bad.shape[0]}/{err.numel()} outside the faithful bound; first got/want/tol: "
                             + ", ".join(f"{i}: {got[i].item():.6g}/{want[i].item():.6g}/{tol[i].item():.3g}"
                                         for i in first))
    frac = (got != want).double().mean().item()
    print(f"[measure] {what}: differ {frac:.6f}, worst err/tol {(err / tol).max().item():.3f}")
    if max_frac is not None:
        assert frac <= max_frac, f"{what}: {frac:.4%} of the elements differ (bound {max_frac:.4%})"
    return frac, (err / tol).max().item()


def act(pre, slope, packed=True):
    """Expected BF16 layer output from the float64 pre-activation acc + bias: bf16 then the packed-BF16 PReLU of
    igemm.cuh, or (packed=False, the x4 strided conv of fused_down.cuh) the fp32 PReLU with the fp32 slope, rounded
    once."""
    s32 = float(torch.tensor(slope, dtype=torch.float32))
    if packed:
        return sb.prelu_packed(sb.round_bf16(pre), s32, float(sb.round_bf16(torch.tensor(s32))))
    return sb.round_bf16(torch.where(pre >= 0, pre, pre * s32))


def ulps(want, packed=True, pre=None):
    """Output ulps a one-ulp difference of the rounded pre-activation can become: two on the negative side of the
    packed PReLU (bf16(s_b * x_b) rounds a second time), one elsewhere.  The side is the pre-activation's: `pre` where
    given; else the sign of `want`, which is the pre-activation's only for slopes >= 0 (a negative slope maps negative
    pre-activations to positive outputs)."""
    if not packed:
        return 1.0
    return torch.where((want if pre is None else pre) < 0, 2.0, 1.0)


def down_faithful(srcs, wt, bt, slope_t, wd, bd, slope_d):
    """The HR half of a feedback group in float64 with the kernels' rounding points (oracle/srfbn_bf16.py): srcs = nsrc
    pairs (map (B,4h,4w,32) of BF16 values, its own sum |w * x| or None) -> (want (B,h,w,32), sum |w * x| through both
    layers, extra tolerance).  H = packed-PReLU(bf16(downtran)) for nsrc > 1; lr = bf16(fp32-PReLU(conv)).  The
    accumulation error of H reaches the output through |wd|, so H's sum |w * x| is carried into the conv's.  H is
    rounded on chip: where its fp32 sum lies next to a BF16 rounding boundary, an element of H (or, in the merged
    kernel, of U before it) rounds the other way, and that one element moves the output by up to 2 ulp(H) * |wd| --
    measured on a B200 at 1 to 8 outputs in a million, 2 to 7 output ulps each.  The extra tolerance allows two such
    elements in each output's 8x8 window.  The maps' device is the computation's."""
    dev = srcs[0][0].device

    def d(t):
        return t.to(dev, torch.float64)

    x = torch.cat([m.permute(0, 3, 1, 2) for m, _ in srcs], dim=1)
    ax = torch.cat([(a if a is not None else torch.zeros_like(m)).permute(0, 3, 1, 2) for m, a in srcs], dim=1)
    if len(srcs) > 1:
        w1 = d(wt).view(32, 32 * len(srcs), 1, 1)
        pre = F.conv2d(x, w1, d(bt))
        ax = F.conv2d(x.abs() + ax, w1.abs(), d(bt).abs())
        x = act(pre, slope_t)
    pre = F.conv2d(x, d(wd), d(bd), stride=4, padding=2)
    absdot = F.conv2d(x.abs() + ax, d(wd).abs(), d(bd).abs(), stride=4, padding=2)
    extra = torch.zeros_like(pre)
    if len(srcs) > 1:
        ulp_h = torch.exp2(torch.floor(torch.log2(x.abs().amax(dim=1, keepdim=True).clamp_min(2.0 ** -126))) - 7)
        win = F.max_pool2d(F.pad(ulp_h, (2, 2, 2, 2)), 8, stride=4)          # the window of each output pixel
        extra = 2 * 2 * win * d(wd).abs().amax(dim=(1, 2, 3)).view(1, 32, 1, 1)
    return (act(pre, slope_d, packed=False).permute(0, 2, 3, 1), absdot.permute(0, 2, 3, 1),
            extra.permute(0, 2, 3, 1))


def bits_equal(got, want, what, dims="b,y,x,c"):
    """Raw-bit equality of two BF16 tensors (-0 and +0 differ); on failure names the first differing elements."""
    a, b = got.view(torch.int16), want.view(torch.int16)
    if torch.equal(a, b):
        return
    idx = (a != b).nonzero().cpu()
    first = [tuple(i.tolist()) for i in idx[:8]]
    pairs = [(got[i].item(), want[i].item()) for i in first]
    raise AssertionError(f"{what}: {idx.shape[0]}/{a.numel()} elements differ; first ({dims}) got/want: "
                         + ", ".join(f"{i}: {g}/{w}" for i, (g, w) in zip(first, pairs)))


def conv_out_abs(hb, x, sd, scale):
    """sum of |terms| of one conv_out output: the conv's |w * x|, |bias|, the skip's |taps| and |add_mean|.  hb (B,32,
    sH,sW) float64 on the computation's device, x (B,3,h,w) and sd anywhere."""
    dev = hb.device

    def d(t):
        return t.to(dev, torch.float64)

    R = sb.Restatement()
    conv = F.conv2d(hb.abs(), R.rb(d(sd["conv_out.0.weight"])).abs(), d(sd["conv_out.0.bias"]).abs(), padding=1)
    xs = (d(x) + d(sd["sub_mean.bias"]).view(1, 3, 1, 1)).abs()
    skip = F.interpolate(xs, scale_factor=scale, mode="bilinear", align_corners=False)
    return conv + skip + d(sd["add_mean.bias"]).abs().view(1, 3, 1, 1)


# ---- the bound plan, one layer range at a time ------------------------------------------------------------------------
def plan_buffer(ent, id, index, shape, dtype):
    """A typed view of activation buffer `id` (BUF_*, `index` of LR / HR) in the workspace of a plan entry of
    SRProjectionModule (ent["plan"], ent["workspace"]); its size must be exactly the shape's."""
    off, n = ctypes.c_size_t(), ctypes.c_size_t()
    _lib.check(_lib.lib().vsr_srfbn_debug_buffer(ent["plan"], id, index, ctypes.byref(off), ctypes.byref(n)),
               f"srfbn_debug_buffer({id}, {index})")
    elems = 1
    for s in shape:
        elems *= s
    itemsize = torch.empty((), dtype=dtype).element_size()
    assert n.value == elems * itemsize, (id, index, n.value, shape, dtype)
    return ent["workspace"][off.value:off.value + n.value].view(dtype).view(shape)


def run_layers(ent, x, first, count):
    """Layers [first, first + count) of the bound plan over its first chunk of the maps x (vsr_srfbn_debug_run_layers),
    on the current stream."""
    _lib.check(_lib.lib().vsr_srfbn_debug_run_layers(ent["plan"], x.data_ptr(), int(first), int(count),
                                                     torch.cuda.current_stream().cuda_stream),
               f"srfbn_debug_run_layers({first}, {count})")
