"""Python front-ends of the single-layer test hooks of the C ABI (vsr_test_*) and the HR block
layout helpers.  Test support only."""
import ctypes

import torch

from video_super_resolution_b200 import _lib


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
