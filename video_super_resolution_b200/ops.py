"""Operator-level Python API over the C ABI (include/vsr_b200.h).

Every function takes CUDA tensors, allocates the outputs (the reference's caller-allocates
convention, resample2d.py:17-19) and enqueues the kernels on torch's current stream.  There is no
CPU path: a non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib

_WORKSPACES: dict = {}


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _req(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: video_super_resolution_b200 ops run on CUDA tensors only (no CPU fallback)")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    # same contract as the reference (`assert input.is_contiguous()`, resample2d.py:10-11)
    if not t.is_contiguous():
        raise ValueError(f"{name}: tensor must be contiguous")
    return t


def _lead(t: torch.Tensor, nd: int, what: str):
    """(lead, windows) of an argument with nd dimensions per window: ((), 1) for one window without a leading
    dimension, ((W,), W) for W >= 1 windows along dim 0."""
    if t.dim() == nd:
        return (), 1
    if t.dim() != nd + 1 or t.shape[0] < 1:
        raise ValueError(what)
    return (t.shape[0],), t.shape[0]


def _workspace(nbytes: int, device) -> torch.Tensor:
    """Caller-side workspace cache (the library itself owns no memory)."""
    key = (device.index, torch.cuda.current_stream().cuda_stream)
    buf = _WORKSPACES.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
        _WORKSPACES[key] = buf
    return buf


def resample2d(input1: torch.Tensor, flow: torch.Tensor, kernel_size: int = 1, bilinear: bool = True) -> torch.Tensor:
    """Reference layout: input1 (B,C,H,W), flow (B,2,H,W) -> (B,C,H,W).
    ref: Resample2dFunction.forward (resample2d.py:8-23), resample2d_kernel.cu:15-72."""
    _req(input1, torch.float32, "input1")
    _req(flow, torch.float32, "input2")
    _, C, _, _ = input1.shape
    B, two, H, W = flow.shape
    if two != 2 or input1.shape[0] != B or tuple(input1.shape[2:]) != (H, W):
        raise ValueError("resample2d: input1 (B,C,H,W) and flow (B,2,H,W) must agree (the reference's only use)")
    out = torch.empty((B, C, H, W), dtype=torch.float32, device=input1.device)
    with torch.cuda.device(input1.device):
        _lib.check(_lib.lib().vsr_resample2d_forward(input1.data_ptr(), flow.data_ptr(), out.data_ptr(), B, C, H, W,
                                                     int(kernel_size), int(bool(bilinear)), _stream()), "resample2d")
    return out


def _deterministic(flag: bool | None) -> bool:
    """None follows torch.use_deterministic_algorithms; True / False force the choice."""
    return torch.are_deterministic_algorithms_enabled() if flag is None else bool(flag)


def _resample2d_backward_into(input1: torch.Tensor, flow: torch.Tensor, grad_output: torch.Tensor,
                             grad_input1: torch.Tensor, grad_input2: torch.Tensor, kernel_size: int = 1,
                             bilinear: bool = True, deterministic: bool | None = None) -> None:
    """Resample2d's backward into caller-allocated gradients (grad_input1 zero-filled, as the reference's caller
    passes it).  deterministic: grad_input1 bit-identical to the CPU restatement instead of fp32 atomics in arrival
    order; None follows torch.are_deterministic_algorithms_enabled()."""
    B, C, H, W = grad_output.shape
    L = _lib.lib()
    with torch.cuda.device(grad_output.device):
        if _deterministic(deterministic):
            ws = _workspace(int(L.vsr_resample2d_backward_deterministic_workspace_bytes(B, H, W)), grad_output.device)
            _lib.check(L.vsr_resample2d_backward_deterministic(
                input1.data_ptr(), flow.data_ptr(), grad_output.data_ptr(), grad_input1.data_ptr(),
                grad_input2.data_ptr(), B, C, H, W, int(kernel_size), int(bool(bilinear)), ws.data_ptr(), ws.numel(),
                _stream()), "resample2d_backward")
        else:
            _lib.check(L.vsr_resample2d_backward(input1.data_ptr(), flow.data_ptr(), grad_output.data_ptr(),
                                                 grad_input1.data_ptr(), grad_input2.data_ptr(), B, C, H, W,
                                                 int(kernel_size), int(bool(bilinear)), _stream()), "resample2d_backward")


def resample2d_backward(input1: torch.Tensor, flow: torch.Tensor, grad_output: torch.Tensor, kernel_size: int = 1,
                        bilinear: bool = True, deterministic: bool | None = None):
    """(grad_input1, grad_input2) of Resample2d.  ref: Resample2dFunction.backward (resample2d.py:25-39).
    deterministic: see _resample2d_backward_into."""
    for t, n in ((input1, "input1"), (flow, "input2"), (grad_output, "grad_output")):
        _req(t, torch.float32, n)
    B, C, H, W = grad_output.shape
    if tuple(input1.shape) != (B, C, H, W) or tuple(flow.shape) != (B, 2, H, W):
        raise ValueError("resample2d_backward: input1/grad_output (B,C,H,W) and flow (B,2,H,W) must agree")
    g1 = torch.zeros_like(input1)                     # the scatter accumulates into it (resample2d.py:32)
    g2 = torch.empty_like(flow)
    _resample2d_backward_into(input1, flow, grad_output, g1, g2, kernel_size, bilinear, deterministic)
    return g1, g2


def channelnorm_backward(x: torch.Tensor, out: torch.Tensor, grad_output: torch.Tensor, norm_deg: int = 2):
    """ref: ChannelNormFunction.backward (channelnorm.py:20-29)."""
    if x.dtype not in _DTYPES:
        raise TypeError(f"input1: expected fp32, fp16 or fp64, got {x.dtype}")
    for t, n in ((x, "input1"), (out, "output"), (grad_output, "grad_output")):
        _req(t, x.dtype, n)
    B, C, H, W = x.shape
    if tuple(out.shape) != (B, 1, H, W) or tuple(grad_output.shape) != (B, 1, H, W):
        raise ValueError("channelnorm_backward: output / grad_output must be (B,1,H,W)")
    g = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().vsr_channelnorm_backward_typed(x.data_ptr(), out.data_ptr(), grad_output.data_ptr(),
                                                             g.data_ptr(), B, C, H, W, int(norm_deg), _DTYPES[x.dtype],
                                                             _stream()), "channelnorm_backward")
    return g


def correlation(input1: torch.Tensor, input2: torch.Tensor, pad_size: int = 3, kernel_size: int = 3,
                max_displacement: int = 20, stride1: int = 1, stride2: int = 2, corr_multiply: int = 1) -> torch.Tensor:
    """FlowNetC cost volume.  ref: CorrelationFunction.forward (correlation.py:9-30)."""
    import ctypes
    _req(input1, torch.float32, "input1")
    _req(input2, torch.float32, "input2")
    if input1.shape != input2.shape or input1.dim() != 4:
        raise ValueError("correlation: two (B,C,H,W) tensors of the same shape expected")
    B, C, H, W = input1.shape
    oc, oh, ow = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    L = _lib.lib()
    _lib.check(L.vsr_correlation_output_shape(C, H, W, pad_size, kernel_size, max_displacement, stride1, stride2,
                                              ctypes.byref(oc), ctypes.byref(oh), ctypes.byref(ow)), "correlation shape")
    out = torch.empty((B, oc.value, oh.value, ow.value), dtype=torch.float32, device=input1.device)
    with torch.cuda.device(input1.device):
        _lib.check(L.vsr_correlation_forward(input1.data_ptr(), input2.data_ptr(), out.data_ptr(), B, C, H, W, pad_size,
                                             kernel_size, max_displacement, stride1, stride2, corr_multiply, _stream()),
                   "correlation")
    return out


def correlation_backward(input1: torch.Tensor, input2: torch.Tensor, grad_output: torch.Tensor, pad_size: int = 3,
                         kernel_size: int = 3, max_displacement: int = 20, stride1: int = 1, stride2: int = 2,
                         corr_multiply: int = 1):
    """(grad_input1, grad_input2) of the cost volume.  ref: CorrelationFunction.backward (correlation.py:32-47)."""
    _req(input1, torch.float32, "input1")
    _req(input2, torch.float32, "input2")
    _req(grad_output, torch.float32, "grad_output")
    if input1.shape != input2.shape or input1.dim() != 4:
        raise ValueError("correlation_backward: two (B,C,H,W) tensors of the same shape expected")
    B, C, H, W = input1.shape
    g1, g2 = torch.empty_like(input1), torch.empty_like(input2)
    with torch.cuda.device(input1.device):
        _lib.check(_lib.lib().vsr_correlation_backward(input1.data_ptr(), input2.data_ptr(), grad_output.data_ptr(),
                                                       g1.data_ptr(), g2.data_ptr(), B, C, H, W, pad_size, kernel_size,
                                                       max_displacement, stride1, stride2, corr_multiply, _stream()),
                   "correlation_backward")
    return g1, g2


def warp(src: torch.Tensor, flow: torch.Tensor, bilinear: bool | int = True, ref: torch.Tensor | None = None):
    """Channels-last warp: src (B,H,W,C), flow (B,H,W,2) -> (B,H,W,C).  With `ref` (B,H,W,C) also
    returns the per-pixel L2 norm of (ref - warped), (B,H,W) (models.py:86-88 fused).
    bilinear: False/0 nearest, True/1 the reference arithmetic bit for bit, 2 fast fp32 (<= 1e-3)."""
    _req(src, torch.float32, "src")
    _req(flow, torch.float32, "flow")
    B, H, W, C = src.shape
    if tuple(flow.shape) != (B, H, W, 2):
        raise ValueError("warp: flow must be (B,H,W,2)")
    dst = torch.empty_like(src)
    norm = None
    if ref is not None:
        _req(ref, torch.float32, "ref")
        if ref.shape != src.shape:
            raise ValueError("warp: ref must have the shape of src")
        norm = torch.empty((B, H, W), dtype=torch.float32, device=src.device)
    with torch.cuda.device(src.device):
        _lib.check(_lib.lib().vsr_warp_nhwc_f32(src.data_ptr(), flow.data_ptr(), dst.data_ptr(),
                                                ref.data_ptr() if ref is not None else None,
                                                norm.data_ptr() if norm is not None else None,
                                                B, H, W, C, int(bilinear), _stream()), "warp")
    return dst if ref is None else (dst, norm)


def warp_window(frames: torch.Tensor, flows: torch.Tensor, centre: int, bilinear: bool | int = 2, want_resid: bool = True):
    """The neighbour warp of a frame window in one launch: frames ([W,]T,H,W,3), flows ([W,]T-1,H,W,2) = one centre ->
    neighbour field per neighbour (frame order, centre left out) -> warped ([W,]T-1,H,W,3) and, with want_resid, the
    per-pixel L2 norm of (frames[centre] - warped[n]) ([W,]T-1,H,W).  With a leading W the one launch warps W windows,
    each to its own centre frame.  No gathered copy of the neighbours, no expanded reference."""
    _req(frames, torch.float32, "frames")
    _req(flows, torch.float32, "flows")
    lead, nw = _lead(frames, 4, "warp_window: frames ([W,]T,H,W,3) expected")
    T, H, W, C = frames.shape[-4:]
    if C != 3 or tuple(flows.shape) != lead + (T - 1, H, W, 2) or not 0 <= centre < T:
        raise ValueError("warp_window: frames ([W,]T,H,W,3), flows ([W,]T-1,H,W,2), 0 <= centre < T expected")
    warped = torch.empty(lead + (T - 1, H, W, 3), dtype=torch.float32, device=frames.device)
    resid = torch.empty(lead + (T - 1, H, W), dtype=torch.float32, device=frames.device) if want_resid else None
    with torch.cuda.device(frames.device):
        _lib.check(_lib.lib().vsr_warp_windows_nhwc3(frames.data_ptr(), flows.data_ptr(), warped.data_ptr(),
                                                     resid.data_ptr() if resid is not None else None, nw, T,
                                                     int(centre), H, W, int(bilinear), _stream()), "warp_window")
    return warped, resid


def compose_flow(g: torch.Tensor | None, f: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """out(p) = g(p) + f(p + g(p)), f sampled bilinearly (border-clamped taps): g maps image A to B, f maps B to C,
    out maps A to C.  g, f, out ([W,]H,W,2); g=None is the identity field (out = f, a copy by our own kernel).  A
    W-window argument may be a view such as x[:, n] of a (W,T-1,H,W,2) array: each window's field is contiguous, and g,
    f and out have one window stride (out=None allocates it with f's strides).  One launch for all windows."""
    lead, nw = _lead(f, 3, "compose_flow: (H,W,2) or (W,H,W,2) fields expected")
    if f.shape[-1] != 2:
        raise ValueError("compose_flow: (H,W,2) or (W,H,W,2) fields expected")
    if out is None:
        out = torch.empty_strided(f.shape, f.stride(), dtype=torch.float32, device=f.device)
    for t, n in ((f, "f"), (g, "g"), (out, "out")):
        if t is not None:
            _req(t[0] if lead else t, torch.float32, n)
            if t.shape != f.shape or (nw > 1 and t.stride(0) != f.stride(0)):
                raise ValueError(f"compose_flow: {n} must have the shape and window stride of f")
    H, W = f.shape[-3:-1]
    with torch.cuda.device(f.device):
        _lib.check(_lib.lib().vsr_compose_flow_windows(g.data_ptr() if g is not None else None, f.data_ptr(),
                                                       out.data_ptr(), nw, f.stride(0) if nw > 1 else 0, H, W,
                                                       _stream()), "compose_flow")
    return out


def warp_labels(labels: torch.Tensor, flow: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """Nearest label warp, bit-exact: labels (B,H,W) u8, flow (B,H,W,2) -> (B,H,W) u8 (written into `out` when
    given).  A contiguous flow is one flat launch over the B images; a view such as x[:, n] of a (B,T-1,H,W,2) array,
    each image's field contiguous, is warped with the image index on the grid."""
    _req(labels, torch.uint8, "labels")
    if labels.dim() != 3 or labels.shape[0] < 1 or tuple(flow.shape) != tuple(labels.shape) + (2,):
        raise ValueError("warp_labels: labels (B,H,W) and flow (B,H,W,2) expected")
    _req(flow[0], torch.float32, "flow")
    B, H, W = labels.shape
    if out is not None:
        _req(out, torch.uint8, "out")
        if out.shape != labels.shape:
            raise ValueError("warp_labels: out must be (B,H,W)")
    dst = torch.empty_like(labels) if out is None else out
    L = _lib.lib()
    with torch.cuda.device(labels.device):
        if flow.is_contiguous():
            _lib.check(L.vsr_warp_labels_u8(labels.data_ptr(), flow.data_ptr(), dst.data_ptr(), B, H, W, _stream()),
                       "warp_labels")
        else:
            _lib.check(L.vsr_warp_labels_u8_windows(labels.data_ptr(), flow.data_ptr(), dst.data_ptr(), B,
                                                    flow.stride(0), H, W, _stream()), "warp_labels")
    return dst

_DTYPES = {torch.float32: 0, torch.float16: 1, torch.float64: 2}     # VSR_DTYPE_*


def channelnorm(x: torch.Tensor, norm_deg: int = 2) -> torch.Tensor:
    """x (B,C,H,W) fp32 / fp16 / fp64 -> (B,1,H,W) of the same dtype.  ref: ChannelNormFunction.forward
    (channelnorm.py:8-18), dtypes of channelnorm_kernel.cu:111."""
    if x.dtype not in _DTYPES:
        raise TypeError(f"input1: expected fp32, fp16 or fp64, got {x.dtype}")
    _req(x, x.dtype, "input1")
    B, C, H, W = x.shape
    out = torch.empty((B, 1, H, W), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().vsr_channelnorm_forward_typed(x.data_ptr(), out.data_ptr(), B, C, H, W, int(norm_deg),
                                                            _DTYPES[x.dtype], _stream()), "channelnorm")
    return out


def project_flow(flow: torch.Tensor, inv_depth: torch.Tensor | None = None, max_disp: float | None = None,
                 deterministic: bool | None = None):
    """Forward flow projection (SURVEY.md Appendix B).  flow (B,h,w,2); inv_depth (B,h,w) or None.
    Returns proj (B,h,w,2) f32, wsum (B,h,w) f32, count (B,h,w) i32, hole (B,h,w) u8.
    max_disp: a promised bound on |fx|, |fy| (<= 8 px) selects the shared-memory tile path; a broken promise is
    detected on the device and costs time, never correctness.  None: no assumption (atomic scatter path).
    deterministic: the sort-and-gather path, bit-identical to the CPU restatement (oracle.or_flow_projection) on every
    run; max_disp is then ignored.  None follows torch.are_deterministic_algorithms_enabled()."""
    _req(flow, torch.float32, "flow")
    B, h, w, two = flow.shape
    if two != 2:
        raise ValueError("project_flow: flow must be (B,h,w,2)")
    if inv_depth is not None:
        _req(inv_depth, torch.float32, "inv_depth")
        if tuple(inv_depth.shape) != (B, h, w):
            raise ValueError("project_flow: inv_depth must be (B,h,w)")
    dev = flow.device
    proj = torch.empty((B, h, w, 2), dtype=torch.float32, device=dev)
    wsum = torch.empty((B, h, w), dtype=torch.float32, device=dev)
    count = torch.empty((B, h, w), dtype=torch.int32, device=dev)
    hole = torch.empty((B, h, w), dtype=torch.uint8, device=dev)
    L = _lib.lib()
    with torch.cuda.device(dev):
        if _deterministic(deterministic):
            ws = _workspace(int(L.vsr_flow_projection_deterministic_workspace_bytes(B, h, w)), dev)
            _lib.check(L.vsr_flow_projection_forward_deterministic(
                flow.data_ptr(), inv_depth.data_ptr() if inv_depth is not None else None, proj.data_ptr(),
                wsum.data_ptr(), count.data_ptr(), hole.data_ptr(), ws.data_ptr(), ws.numel(), B, h, w, _stream()),
                "project_flow")
            return proj, wsum, count, hole
        nbytes = int(L.vsr_flow_projection_workspace_bytes(B, h, w))
        ws = _workspace(nbytes, dev)
        _lib.check(L.vsr_flow_projection_forward_bounded(
            flow.data_ptr(), inv_depth.data_ptr() if inv_depth is not None else None, proj.data_ptr(), wsum.data_ptr(),
            count.data_ptr(), hole.data_ptr(), ws.data_ptr(), ws.numel(), B, h, w,
            -1.0 if max_disp is None else float(max_disp), _stream()), "project_flow")
    return proj, wsum, count, hole


def project_depth_flow(flow: torch.Tensor, inv_depth: torch.Tensor, max_disp: float | None = None,
                       deterministic: bool | None = None):
    """Inverse-depth-weighted projection (nearer surfaces dominate contested targets)."""
    if inv_depth is None:
        raise ValueError("project_depth_flow: inv_depth is required")
    return project_flow(flow, inv_depth, max_disp, deterministic)


def flow_to_image(flow: torch.Tensor, out_size=None, want_u8: bool = True):
    """Middlebury colour code of one flow map, on the device.  flow (h,w,2) f32 -> (img, planes):
    img (h,w,3) u8 (None unless want_u8), planes (3,H,W) f32 = the image transposed to CHW and nearest-resized to
    out_size=(H,W) (None unless out_size is given).
    ref: utils/flow_utils.py:4-24 via FlowProjectionModule.py:31-32; video_super_resolution.py:35,52."""
    _req(flow, torch.float32, "flow")
    if flow.dim() != 3 or flow.shape[2] != 2:
        raise ValueError("flow_to_image: (h,w,2) flow expected")
    if out_size is None and not want_u8:
        raise ValueError("flow_to_image: nothing to compute")
    h, w = flow.shape[:2]
    img = torch.empty((h, w, 3), dtype=torch.uint8, device=flow.device) if want_u8 else None
    planes = torch.empty((3, int(out_size[0]), int(out_size[1])), dtype=torch.float32, device=flow.device) \
        if out_size is not None else None
    ws = torch.empty(2, dtype=torch.int32, device=flow.device)
    with torch.cuda.device(flow.device):
        _lib.check(_lib.lib().vsr_flow_to_image(flow.data_ptr(), h, w, img.data_ptr() if want_u8 else None,
                                                planes.data_ptr() if planes is not None else None,
                                                planes.shape[1] if planes is not None else 0,
                                                planes.shape[2] if planes is not None else 0,
                                                ws.data_ptr(), _stream()), "flow_to_image")
    return img, planes


def vos_threshold(logits_a: torch.Tensor, logits_b: torch.Tensor) -> torch.Tensor:
    """sigmoid(a)+sigmoid(b) > 0.7 -> u8 {0,1}: logits ([W,]h,w) x2 -> mask ([W,]h,w), one launch for all windows.
    ref: VOSProjectionModule.py:22-25."""
    _req(logits_a, torch.float32, "logits_a")
    _req(logits_b, torch.float32, "logits_b")
    _, nw = _lead(logits_a, 2, "vos_threshold: two ([W,]h,w) tensors expected")
    if logits_b.shape != logits_a.shape:
        raise ValueError("vos_threshold: two ([W,]h,w) tensors expected")
    h, w = logits_a.shape[-2:]
    mask = torch.empty(logits_a.shape, dtype=torch.uint8, device=logits_a.device)
    with torch.cuda.device(logits_a.device):
        _lib.check(_lib.lib().vsr_vos_threshold_windows(logits_a.data_ptr(), logits_b.data_ptr(), mask.data_ptr(), nw,
                                                        h, w, _stream()), "vos_threshold")
    return mask


def mask_fill(image: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """image (C,h,w) f32, mask (h,w) u8 -> image with masked pixels zeroed.
    ref: video_super_resolution.py:58-60 (MaskedArray(..., fill_value=0).filled())."""
    _req(image, torch.float32, "image")
    _req(mask, torch.uint8, "mask")
    C, h, w = image.shape
    if tuple(mask.shape) != (h, w):
        raise ValueError("mask_fill: mask must be (h,w)")
    out = torch.empty_like(image)
    with torch.cuda.device(image.device):
        _lib.check(_lib.lib().vsr_mask_fill(image.data_ptr(), mask.data_ptr(), out.data_ptr(), C, h, w, _stream()),
                   "mask_fill")
    return out


def assemble_stack(warped: torch.Tensor, frames: torch.Tensor, proj: torch.Tensor, resid: torch.Tensor,
                   depth: torch.Tensor, estimate: torch.Tensor | None, centre_idx: int,
                   out: torch.Tensor | None = None) -> torch.Tensor:
    """One-pass assembly of the ([W,]3T-1,3,h,w) map stack (video_super_resolution.py:33-40), one launch for all
    windows.  warped ([W,]T-1,h,w,3), frames ([W,]T,h,w,3), proj ([W,]T-1,h,w,2), resid / depth ([W,]T-1,h,w),
    estimate ([W,]3,h,w) | None.  The centre frame and, without an estimate, LR frame 0 of each window (the
    reference's `else data_clone[0:1]`, :37-38) are read from frames in place."""
    for t, n in ((warped, "warped"), (frames, "frames"), (proj, "proj"), (resid, "resid"), (depth, "depth")):
        _req(t, torch.float32, n)
    lead, nw = _lead(frames, 4, "assemble_stack: frames ([W,]T,h,w,3) expected")
    T, h, w, C = frames.shape[-4:]
    if C != 3 or tuple(warped.shape) != lead + (T - 1, h, w, 3) or tuple(proj.shape) != lead + (T - 1, h, w, 2) or \
            tuple(resid.shape) != lead + (T - 1, h, w) or tuple(depth.shape) != lead + (T - 1, h, w) or \
            not 0 <= centre_idx < T:
        raise ValueError("assemble_stack: inconsistent shapes")
    if estimate is not None:
        _req(estimate, torch.float32, "estimate")
        if tuple(estimate.shape) != lead + (3, h, w):
            raise ValueError("assemble_stack: estimate must be ([W,]3,h,w)")
    if out is None:
        out = torch.empty(lead + (3 * T - 1, 3, h, w), dtype=torch.float32, device=warped.device)
    else:
        _req(out, torch.float32, "out")
        if tuple(out.shape) != lead + (3 * T - 1, 3, h, w):
            raise ValueError("assemble_stack: out must be ([W,]3T-1,3,h,w)")
    with torch.cuda.device(warped.device):
        _lib.check(_lib.lib().vsr_assemble_stack_windows(
            warped.data_ptr(), frames.select(-4, centre_idx).data_ptr(), proj.data_ptr(), resid.data_ptr(),
            depth.data_ptr(), estimate.data_ptr() if estimate is not None else None, frames.data_ptr(), out.data_ptr(),
            nw, T * h * w * 3, T, int(centre_idx), h, w, _stream()), "assemble_stack")
    return out


def estimate_slot(hr: torch.Tensor, mask: torch.Tensor | None, slot: torch.Tensor, scale: int = 4) -> torch.Tensor:
    """slot ([W,]3,h,w) <- nearest-downsized hr ([W,]3,h*scale,w*scale) with the pixels of mask ([W,]h,w) zeroed
    (video_super_resolution.py:44,58-60), one launch for all windows.  `slot` is written in place: a view of the
    stack, such as stack[:, M-1] of a (W,M,3,h,w) stack, with each window's slot contiguous."""
    _req(hr, torch.float32, "hr")
    lead, nw = _lead(slot, 3, "estimate_slot: slot ([W,]3,h,w) expected")
    _req(slot[0] if lead else slot, torch.float32, "slot")
    c, h, w = slot.shape[-3:]
    if c != 3 or tuple(hr.shape) != lead + (3, h * scale, w * scale):
        raise ValueError("estimate_slot: slot ([W,]3,h,w) and hr ([W,]3,h*scale,w*scale) expected")
    if mask is not None:
        _req(mask, torch.uint8, "mask")
        if tuple(mask.shape) != lead + (h, w):
            raise ValueError("estimate_slot: mask must be ([W,]h,w)")
    with torch.cuda.device(hr.device):
        _lib.check(_lib.lib().vsr_estimate_slot_windows(hr.data_ptr(), mask.data_ptr() if mask is not None else None,
                                                        slot.data_ptr(), nw, slot.stride(0) if nw > 1 else 0, h, w,
                                                        int(scale), _stream()), "estimate_slot")
    return slot


def unpack_bands(src: torch.Tensor, dst: torch.Tensor, bounds, planes: int, row: int, band_stride: int) -> torch.Tensor:
    """The reorder after a gather of row bands (vsr_unpack_bands): src holds len(bounds)-1 bands band_stride elements
    apart (0: back to back), band p `planes` planes of bounds[p+1]-bounds[p] rows of `row` elements; dst (planes,
    bounds[-1], row) receives band p at rows [bounds[p], bounds[p+1]) of every plane.  fp32 or u8 tensors; returns dst."""
    if src.dtype != dst.dtype or src.dtype not in (torch.float32, torch.uint8):
        raise TypeError("unpack_bands: src and dst must both be float32 or both uint8")
    _req(src, src.dtype, "src")
    _req(dst, dst.dtype, "dst")
    G = len(bounds) - 1
    need = band_stride * (G - 1) + planes * (bounds[-1] - bounds[-2]) * row if band_stride else dst.numel()
    if dst.numel() != planes * bounds[-1] * row or src.numel() < need:
        raise ValueError("unpack_bands: buffer sizes do not match the band geometry")
    b = (ctypes.c_int * (G + 1))(*bounds)
    with torch.cuda.device(dst.device):
        _lib.check(_lib.lib().vsr_unpack_bands(src.data_ptr(), dst.data_ptr(), src.element_size(), int(planes), int(row),
                                               b, G, int(band_stride), _stream()), "unpack_bands")
    return dst
