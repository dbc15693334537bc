"""ctypes front-end of the CPU oracle (oracle/oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package never imports this module.

All functions take and return numpy arrays; layouts are stated per function.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")
_lib = None

_f32p = ctypes.POINTER(ctypes.c_float)
_u8p = ctypes.POINTER(ctypes.c_uint8)
_i32p = ctypes.POINTER(ctypes.c_int32)


def build(force: bool = False) -> str:
    """Compile oracle.c with gcc (recipe: oracle/Makefile)."""
    src = os.path.join(_HERE, "oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "all"])
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_LIB_PATH)
        L = ctypes.c_long
        I = ctypes.c_int
        _lib.or_resample2d.argtypes = [_f32p, _f32p, _f32p, I, I, I, I] + [L] * 12 + [I, I, I, I]
        _lib.or_resample2d.restype = None
        _lib.or_warp_nhwc_fast.argtypes = [_f32p] * 5 + [I] * 6
        _lib.or_warp_nhwc_fast.restype = None
        _lib.or_compose_flow_fast.argtypes = [_f32p] * 3 + [I] * 4
        _lib.or_compose_flow_fast.restype = None
        _lib.or_warp_labels.argtypes = [_u8p, _f32p, _u8p, I, I, I]
        _lib.or_warp_labels.restype = None
        _lib.or_channelnorm.argtypes = [_f32p, _f32p, I, I, I, I, L, L, L, L]
        _lib.or_channelnorm.restype = None
        _lib.or_flow_projection.argtypes = [_f32p, _f32p, _f32p, _f32p, _i32p, _u8p, I, I, I]
        _lib.or_flow_projection.restype = None
        _lib.or_vos_threshold.argtypes = [_f32p, _f32p, _u8p, L]
        _lib.or_vos_threshold.restype = None
        _lib.or_mask_fill.argtypes = [_f32p, _u8p, _f32p, I, L]
        _lib.or_mask_fill.restype = None
        _lib.or_resample2d_backward.argtypes = [_f32p] * 5 + [I, I, I, I]
        _lib.or_resample2d_backward.restype = None
        _lib.or_channelnorm_backward.argtypes = [_f32p] * 4 + [I, I, L]
        _lib.or_channelnorm_backward.restype = None
        _lib.or_correlation.argtypes = [_f32p] * 3 + [I] * 14
        _lib.or_correlation.restype = None
        _lib.or_correlation_backward.argtypes = [_f32p] * 3 + [I] * 11
        _lib.or_correlation_backward.restype = None
        _lib.or_correlation_backward_chain.argtypes = [_f32p] * 3 + [I] * 13
        _lib.or_correlation_backward_chain.restype = None
        _lib.or_flow2img.argtypes = [_f32p, _u8p, I, I]
        _lib.or_flow2img.restype = None
        _lib.or_resize_nearest_planar.argtypes = [_u8p, _f32p, I, I, I, I]
        _lib.or_resize_nearest_planar.restype = None
    return _lib


def _p(a, t):
    return a.ctypes.data_as(t)


def _c(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _fan_rows(fn, H, threads):
    """Run fn(y0, y1) over `threads` row ranges (ctypes drops the GIL during the C call)."""
    threads = max(1, min(int(threads), H))
    if threads == 1:
        fn(0, H)
        return
    edges = np.linspace(0, H, threads + 1).astype(int)
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda i: fn(int(edges[i]), int(edges[i + 1])), range(threads)))


def resample2d_nchw(input1, flow, kernel_size=1, bilinear=True, threads=1):
    """Reference layout: input1 (B,C,H,W), flow (B,2,H,W) -> (B,C,H,W).
    ref: resample2d.py:8-23, resample2d_kernel.cu:15-72."""
    input1 = _c(input1, np.float32)
    flow = _c(flow, np.float32)
    B, C, H, W = input1.shape
    assert flow.shape == (B, 2, H, W)
    out = np.zeros((B, C, H, W), np.float32)
    L = lib()

    def run(y0, y1):
        L.or_resample2d(_p(input1, _f32p), _p(flow, _f32p), _p(out, _f32p), B, C, H, W,
                        C * H * W, H * W, W, 1, 2 * H * W, H * W, W, 1, C * H * W, H * W, W, 1,
                        int(kernel_size), int(bool(bilinear)), y0, y1)

    _fan_rows(run, H, threads)
    return out


def warp_nhwc(src, flow, bilinear=True, threads=1, ref=None):
    """Pipeline layout: src (B,H,W,C), flow (B,H,W,2) -> (B,H,W,C).  bilinear: False/0 nearest, True/1 the reference
    arithmetic, 2 the fast mode (or_warp_nhwc_fast: fp32 FMA blend).  With ref (B,H,W,C) also returns the per-pixel
    L2 norm of (ref - warped), (B,H,W), as ops.warp(..., ref=ref)."""
    src = _c(src, np.float32)
    flow = _c(flow, np.float32)
    B, H, W, C = src.shape
    assert flow.shape == (B, H, W, 2)
    out = np.zeros((B, H, W, C), np.float32)
    L = lib()
    mode = int(bilinear)
    if mode == 2:
        if ref is not None:
            ref = _c(ref, np.float32)
            assert ref.shape == src.shape
        norm = np.zeros((B, H, W), np.float32) if ref is not None else None

        def run(y0, y1):
            L.or_warp_nhwc_fast(_p(src, _f32p), _p(flow, _f32p), _p(out, _f32p),
                                _p(ref, _f32p) if ref is not None else None,
                                _p(norm, _f32p) if ref is not None else None, B, H, W, C, y0, y1)

        _fan_rows(run, H, threads)
        return out if ref is None else (out, norm)
    assert mode in (0, 1), bilinear

    def run(y0, y1):
        L.or_resample2d(_p(src, _f32p), _p(flow, _f32p), _p(out, _f32p), B, C, H, W,
                        H * W * C, 1, W * C, C, H * W * 2, 1, W * 2, 2, H * W * C, 1, W * C, C,
                        1, mode, y0, y1)

    _fan_rows(run, H, threads)
    return out if ref is None else (out, channelnorm_nhwc(_c(ref, np.float32) - out))


def warp_labels(labels, flow):
    """labels (B,H,W) u8, flow (B,H,W,2) -> (B,H,W) u8.  ref: resample2d_kernel.cu:65-70."""
    labels = _c(labels, np.uint8)
    flow = _c(flow, np.float32)
    B, H, W = labels.shape
    out = np.zeros((B, H, W), np.uint8)
    lib().or_warp_labels(_p(labels, _u8p), _p(flow, _f32p), _p(out, _u8p), B, H, W)
    return out


def channelnorm_nchw(x):
    """x (B,C,H,W) -> (B,1,H,W).  ref: channelnorm_kernel.cu:19-60."""
    x = _c(x, np.float32)
    B, C, H, W = x.shape
    out = np.zeros((B, 1, H, W), np.float32)
    lib().or_channelnorm(_p(x, _f32p), _p(out, _f32p), B, C, H, W, C * H * W, H * W, W, 1)
    return out


def channelnorm_nhwc(x):
    """x (B,H,W,C) -> (B,H,W)."""
    x = _c(x, np.float32)
    B, H, W, C = x.shape
    out = np.zeros((B, H, W), np.float32)
    lib().or_channelnorm(_p(x, _f32p), _p(out, _f32p), B, C, H, W, H * W * C, 1, W * C, C)
    return out


def resample2d_backward(input1, flow, grad_output):
    """(grad_input1, grad_input2), NCHW.  ref: resample2d_kernel.cu:75-198, resample2d.py:25-39."""
    input1 = _c(input1, np.float32)
    flow = _c(flow, np.float32)
    grad_output = _c(grad_output, np.float32)
    B, C, H, W = input1.shape
    g1 = np.zeros_like(input1)
    g2 = np.zeros_like(flow)
    lib().or_resample2d_backward(_p(input1, _f32p), _p(flow, _f32p), _p(grad_output, _f32p), _p(g1, _f32p), _p(g2, _f32p),
                                 B, C, H, W)
    return g1, g2


def channelnorm_backward(x, out, grad_output):
    """ref: channelnorm_kernel.cu:64-96."""
    x = _c(x, np.float32)
    out = _c(out, np.float32)
    grad_output = _c(grad_output, np.float32)
    B, C, H, W = x.shape
    g = np.zeros_like(x)
    lib().or_channelnorm_backward(_p(x, _f32p), _p(out, _f32p), _p(grad_output, _f32p), _p(g, _f32p), B, C, H * W)
    return g


def correlation(input1, input2, pad_size=3, kernel_size=3, max_displacement=20, stride1=1, stride2=2, padded=False,
                items=None, threads=1):
    """FlowNetC cost volume, NCHW.  ref: correlation_cuda.cc:25-42, correlation_cuda_kernel.cu:73-147.
    padded=True: the reference's zero padding with every product taken (the kernels' rule, NaN from 0 * Inf);
    padded=False: taps with a position outside the image skipped.  items=(n0, n1) restates batch items n0..n1-1 only
    (the result has n1 - n0 items); threads fans the output rows out."""
    input1 = _c(input1, np.float32)
    input2 = _c(input2, np.float32)
    if items is not None:
        input1, input2 = input1[items[0]:items[1]], input2[items[0]:items[1]]
    B, C, H, W = input1.shape
    border = (kernel_size - 1) // 2 + max_displacement
    outH = -(-(H + 2 * pad_size - 2 * border) // stride1)
    outW = -(-(W + 2 * pad_size - 2 * border) // stride1)
    D = 2 * (max_displacement // stride2) + 1
    out = np.zeros((B, D * D, outH, outW), np.float32)
    L = lib()
    _fan_rows(lambda y0, y1: L.or_correlation(_p(input1, _f32p), _p(input2, _f32p), _p(out, _f32p), B, C, H, W, pad_size,
                                              kernel_size, max_displacement, stride1, stride2, outH, outW, int(padded),
                                              y0, y1), outH, threads)
    return out


def flow_projection(flow, inv_depth=None, threads=1):
    """flow (B,h,w,2), inv_depth (B,h,w)|None -> proj (B,h,w,2), wsum (B,h,w), count i32, hole u8.
    SURVEY.md Appendix B (PARITY UNPINNED: no reference implementation exists)."""
    flow = _c(flow, np.float32)
    B, h, w, two = flow.shape
    assert two == 2
    if inv_depth is not None:
        inv_depth = _c(inv_depth, np.float32)
        assert inv_depth.shape == (B, h, w)
    proj = np.zeros((B, h, w, 2), np.float32)
    wsum = np.zeros((B, h, w), np.float32)
    count = np.zeros((B, h, w), np.int32)
    hole = np.zeros((B, h, w), np.uint8)
    L = lib()

    def one(b):
        L.or_flow_projection(_p(flow[b:b + 1], _f32p),
                             _p(inv_depth[b:b + 1], _f32p) if inv_depth is not None else None,
                             _p(proj[b:b + 1], _f32p), _p(wsum[b:b + 1], _f32p),
                             _p(count[b:b + 1], _i32p), _p(hole[b:b + 1], _u8p), 1, h, w)

    threads = max(1, min(int(threads), B))
    if threads == 1:
        for b in range(B):
            one(b)
    else:
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(one, range(B)))
    return proj, wsum, count, hole


def vos_threshold(logits_a, logits_b):
    """(h,w) f32 x2 -> (h,w) u8.  ref: VOSProjectionModule.py:22-25."""
    a = _c(logits_a, np.float32)
    b = _c(logits_b, np.float32)
    out = np.zeros(a.shape, np.uint8)
    lib().or_vos_threshold(_p(a, _f32p), _p(b, _f32p), _p(out, _u8p), a.size)
    return out


def mask_fill(image, mask):
    """image (C,h,w) f32, mask (h,w) u8 -> (C,h,w).  ref: video_super_resolution.py:58-60."""
    image = _c(image, np.float32)
    mask = _c(mask, np.uint8)
    C = image.shape[0]
    out = np.zeros_like(image)
    lib().or_mask_fill(_p(image, _f32p), _p(mask, _u8p), _p(out, _f32p), C, mask.size)
    return out


def assemble_stack(warped, centre, proj, resid, depth, estimate, centre_idx, fallback=None):
    """numpy restatement of the stack assembly (video_super_resolution.py:33-40 generalised to T
    frames): warped (T-1,h,w,3), centre (h,w,3), proj (T-1,h,w,2), resid/depth (T-1,h,w),
    estimate (3,h,w)|None -> (3T-1,3,h,w).  Without an estimate the last slot is `fallback` (h,w,3) = LR frame 0
    of the window (:37-38 `else data_clone[0:1]`)."""
    if fallback is None:
        fallback = centre
    Tm1, h, w, _ = warped.shape
    T = Tm1 + 1
    out = np.zeros((3 * T - 1, 3, h, w), np.float32)
    n = 0
    for t in range(T):
        if t == centre_idx:
            out[t] = centre.transpose(2, 0, 1)                       # transpose1201
        else:
            out[t] = warped[n].transpose(2, 0, 1)
            n += 1
    for n in range(Tm1):
        out[T + n, 0] = proj[n, :, :, 0]
        out[T + n, 1] = proj[n, :, :, 1]
        out[T + n, 2] = resid[n]
        out[2 * T - 1 + n] = np.stack((depth[n],) * 3)               # maskprocess
    out[3 * T - 2] = fallback.transpose(2, 0, 1) if estimate is None else estimate
    return out


def compose_flow(g, f, fast=False, threads=1):
    """out(p) = g(p) + f(p + g(p)), f (h,w,2) sampled with the Resample2d taps and border rule (Appendix A);
    g maps image A to B, f maps B to C, the result maps A to C.  fast=True: the arithmetic of ops.compose_flow
    (compose_flow_kernel: fast-mode blend, fp32 add of g), g=None the identity field; fast=False: the exact blend."""
    f = _c(f, np.float32)
    if not fast:
        g = _c(g, np.float32)
        return (g + warp_nhwc(f[None], g[None], True)[0]).astype(np.float32)
    H, W, two = f.shape
    assert two == 2
    if g is not None:
        g = _c(g, np.float32)
        assert g.shape == f.shape
    out = np.zeros_like(f)
    L = lib()
    _fan_rows(lambda y0, y1: L.or_compose_flow_fast(_p(g, _f32p) if g is not None else None, _p(f, _f32p),
                                                    _p(out, _f32p), H, W, y0, y1), H, threads)
    return out


def chain_flows(proj, flows, centre, fast=False, threads=1):
    """Centre -> neighbour flows (T-1,h,w,2), frame order with the centre left out (WarpFusePipeline docstring):
    past frames chain the PROJECTED flows (they live in the later frame's coordinates), future frames the forward
    flows (they live in the earlier frame's).  fast=True restates WarpFusePipeline.chain_flows link for link, the
    first link of each side included (compose_flow(None, .), a copy up to the sign of zero)."""
    Tm1 = flows.shape[0]
    T, c = Tm1 + 1, centre
    G = np.zeros_like(flows)

    def link(g, f):
        return compose_flow(g, f, fast=fast, threads=threads)

    G[c - 1] = link(None, proj[c - 1]) if fast else proj[c - 1]
    for t in range(c - 2, -1, -1):
        G[t] = link(G[t + 1], proj[t])
    if c + 1 < T:
        G[c] = link(None, flows[c]) if fast else flows[c]
        for t in range(c + 2, T):
            G[t - 1] = link(G[t - 2], flows[t - 1])
    return G


def estimate_slot(hr, mask, scale=4):
    """hr (3,H,W) -> (3,h,w): nearest downsize (F.interpolate default: src = dst*scale,
    video_super_resolution.py:44) then MaskedArray(..., fill_value=0).filled() (:58-60)."""
    lo = np.ascontiguousarray(hr[:, ::scale, ::scale], dtype=np.float32)
    if mask is not None:
        lo = np.ma.MaskedArray(lo, np.stack((mask,) * 3).astype(bool), fill_value=0).filled()
    return lo.astype(np.float32)


def warp_fuse_front(frames, flows, inv_depth, logits_a, logits_b, estimate=None, threads=1, fast=False, projected=None):
    """CPU restatement of WarpFusePipeline.project_and_warp (a1-a5 + a7): returns the map stack and
    the intermediates.  frames (T,h,w,3), flows (T-1,h,w,2), inv_depth (T-1,h,w), logits (h,w) x2.
    fast=False: the warps and the flow chain in the reference's exact arithmetic; fast=True: in the arithmetic the
    pipeline runs (mode 2 warp with the fused residual, compose_flow_kernel), so that with the deterministic projection
    every output is restated bit for bit.
    projected: (proj_flow, proj_depth, wsum) taken as given instead of this restatement's projections -- the chain,
    warps, label warp and assembly downstream of them are restated from those arrays.
    W windows: frames (W,T,h,w,3) and every other input with the same leading W (estimate (W,3,h,w) | None,
    projected arrays (W,T-1,...)): one restatement per window, results stacked along a leading W."""
    frames = np.asarray(frames)
    if frames.ndim == 5:
        outs = [warp_fuse_front(frames[b], flows[b], inv_depth[b], logits_a[b], logits_b[b],
                                None if estimate is None else estimate[b], threads, fast,
                                None if projected is None else tuple(p[b] for p in projected))
                for b in range(frames.shape[0])]
        return (np.stack([o[0] for o in outs]), {k: np.stack([o[1][k] for o in outs]) for k in outs[0][1]})
    T = frames.shape[0]
    c = T // 2
    proj_f, _, cnt_f, hole_f = flow_projection(flows, None, threads=threads)
    proj_d, wsum, cnt_d, hole_d = flow_projection(flows, inv_depth, threads=threads)
    if projected is not None:
        proj_f, proj_d, wsum = (_c(p, np.float32) for p in projected)
    G = chain_flows(proj_d, flows, c, fast=fast, threads=threads)
    neigh = np.ascontiguousarray(frames[[t for t in range(T) if t != c]])
    centre = np.broadcast_to(frames[c], neigh.shape)
    warped, resid = warp_nhwc(neigh, G, 2 if fast else True, threads=threads, ref=centre)
    mask = vos_threshold(logits_a, logits_b)
    mask_w = warp_labels(mask[None], G[c - 1][None])[0]
    stack = assemble_stack(warped, frames[c], proj_f, resid, wsum, estimate, c, fallback=frames[0])
    return stack, {"proj_flow": proj_f, "count_flow": cnt_f, "hole_flow": hole_f, "proj_depth": proj_d, "wsum": wsum,
                   "count_depth": cnt_d, "hole_depth": hole_d, "warped": warped, "resid": resid, "mask": mask,
                   "mask_warped": mask_w, "centre_flows": G}


def flow2img(flow):
    """utils/flow_utils.py:4-24: flow (h,w,2) fp32 -> Middlebury colour code (h,w,3) u8."""
    flow = _c(flow, np.float32)
    h, w = flow.shape[:2]
    img = np.empty((h, w, 3), np.uint8)
    lib().or_flow2img(_p(flow, _f32p), _p(img, _u8p), h, w)
    return img


def resize_nearest_planar(img, H, W):
    """interpolate(transpose1323(img), (H,W)) (video_super_resolution.py:35): (h,w,3) u8 -> (3,H,W) fp32."""
    img = _c(img, np.uint8)
    h, w = img.shape[:2]
    out = np.empty((3, H, W), np.float32)
    lib().or_resize_nearest_planar(_p(img, _u8p), _p(out, _f32p), h, w, H, W)
    return out


def correlation_backward(input1, input2, grad_output, pad_size, kernel_size, max_displacement, stride2):
    """correlation_cuda.backward with stride1 = 1 (correlation_cuda_kernel.cu:148-333): (grad_input1, grad_input2)."""
    a, b, g = _c(input1, np.float32), _c(input2, np.float32), _c(grad_output, np.float32)
    B, C, H, W = a.shape
    oh, ow = g.shape[2], g.shape[3]
    g1, g2 = np.empty_like(a), np.empty_like(a)
    lib().or_correlation_backward(_p(b, _f32p), _p(g, _f32p), _p(g1, _f32p), 0, B, C, H, W, pad_size, kernel_size,
                                  max_displacement, stride2, oh, ow)
    lib().or_correlation_backward(_p(a, _f32p), _p(g, _f32p), _p(g2, _f32p), 1, B, C, H, W, pad_size, kernel_size,
                                  max_displacement, stride2, oh, ow)
    return g1, g2


def correlation_backward_chain(input1, input2, grad_output, pad_size, kernel_size, max_displacement, stride2,
                               items=None, channels=None, threads=1):
    """(grad_input1, grad_input2) in the order of correlation_backward_kernel: one fmaf chain per element over (tj, ti,
    j, i), padded values zero with their products taken.  items=(n0, n1) / channels=(c0, c1) restate that block only
    (the results are (n1 - n0, c1 - c0, H, W)); threads fans the channels out."""
    a, b, g = _c(input1, np.float32), _c(input2, np.float32), _c(grad_output, np.float32)
    if items is not None:
        a, b, g = a[items[0]:items[1]], b[items[0]:items[1]], g[items[0]:items[1]]
    B, C, H, W = a.shape
    oh, ow = g.shape[2], g.shape[3]
    c0, c1 = channels if channels is not None else (0, C)
    g1, g2 = np.zeros_like(a), np.zeros_like(a)
    L = lib()

    def run(k0, k1):
        for which, other, gin in ((0, b, g1), (1, a, g2)):
            L.or_correlation_backward_chain(_p(other, _f32p), _p(g, _f32p), _p(gin, _f32p), which, B, C, H, W, pad_size,
                                            kernel_size, max_displacement, stride2, oh, ow, c0 + k0, c0 + k1)

    _fan_rows(run, c1 - c0, threads)
    return np.ascontiguousarray(g1[:, c0:c1]), np.ascontiguousarray(g2[:, c0:c1])
