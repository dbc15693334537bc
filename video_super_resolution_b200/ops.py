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
    """The neighbour warp of one window in one launch: frames (T,H,W,3), flows (T-1,H,W,2) = one centre -> neighbour
    field per neighbour (frame order, centre left out) -> warped (T-1,H,W,3) and, with want_resid, the per-pixel L2
    norm of (frames[centre] - warped[n]) (T-1,H,W).  No gathered copy of the neighbours, no expanded reference."""
    _req(frames, torch.float32, "frames")
    _req(flows, torch.float32, "flows")
    T, H, W, C = frames.shape
    if C != 3 or tuple(flows.shape) != (T - 1, H, W, 2) or not 0 <= centre < T:
        raise ValueError("warp_window: frames (T,H,W,3), flows (T-1,H,W,2), 0 <= centre < T expected")
    warped = torch.empty((T - 1, H, W, 3), dtype=torch.float32, device=frames.device)
    resid = torch.empty((T - 1, H, W), dtype=torch.float32, device=frames.device) if want_resid else None
    with torch.cuda.device(frames.device):
        _lib.check(_lib.lib().vsr_warp_window_nhwc3(frames.data_ptr(), flows.data_ptr(), warped.data_ptr(),
                                                    resid.data_ptr() if resid is not None else None, T, int(centre), H, W,
                                                    int(bilinear), _stream()), "warp_window")
    return warped, resid


def compose_flow(g: torch.Tensor, f: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """out(p) = g(p) + f(p + g(p)), f sampled bilinearly (border-clamped taps): g maps image A to B, f maps B to C,
    out maps A to C.  g, f (B,H,W,2) or (H,W,2); g=None is the identity field (out = f, a copy by our own kernel)."""
    _req(f, torch.float32, "f")
    if g is not None:
        _req(g, torch.float32, "g")
    if (g is not None and g.shape != f.shape) or f.shape[-1] != 2 or f.dim() not in (3, 4):
        raise ValueError("compose_flow: two (B,H,W,2) or (H,W,2) fields of the same shape expected")
    B = f.shape[0] if f.dim() == 4 else 1
    H, W = f.shape[-3], f.shape[-2]
    if out is None:
        out = torch.empty_like(f)
    else:
        _req(out, torch.float32, "out")
        if out.shape != f.shape:
            raise ValueError("compose_flow: out must have the shape of f")
    with torch.cuda.device(f.device):
        _lib.check(_lib.lib().vsr_compose_flow(g.data_ptr() if g is not None else None, f.data_ptr(), out.data_ptr(),
                                               B, H, W, _stream()), "compose_flow")
    return out


def warp_labels(labels: torch.Tensor, flow: torch.Tensor) -> torch.Tensor:
    """Nearest label warp: labels (B,H,W) u8, flow (B,H,W,2) -> (B,H,W) u8, bit-exact."""
    _req(labels, torch.uint8, "labels")
    _req(flow, torch.float32, "flow")
    B, H, W = labels.shape
    if tuple(flow.shape) != (B, H, W, 2):
        raise ValueError("warp_labels: flow must be (B,H,W,2)")
    dst = torch.empty_like(labels)
    with torch.cuda.device(labels.device):
        _lib.check(_lib.lib().vsr_warp_labels_u8(labels.data_ptr(), flow.data_ptr(), dst.data_ptr(), B, H, W,
                                                 _stream()), "warp_labels")
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
    """sigmoid(a)+sigmoid(b) > 0.7 -> u8 {0,1}.  ref: VOSProjectionModule.py:22-25."""
    _req(logits_a, torch.float32, "logits_a")
    _req(logits_b, torch.float32, "logits_b")
    if logits_a.shape != logits_b.shape or logits_a.dim() != 2:
        raise ValueError("vos_threshold: two (h,w) tensors expected")
    h, w = logits_a.shape
    mask = torch.empty((h, w), dtype=torch.uint8, device=logits_a.device)
    with torch.cuda.device(logits_a.device):
        _lib.check(_lib.lib().vsr_vos_threshold(logits_a.data_ptr(), logits_b.data_ptr(), mask.data_ptr(), h, w,
                                                _stream()), "vos_threshold")
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


def assemble_stack(warped: torch.Tensor, centre: torch.Tensor, proj: torch.Tensor, resid: torch.Tensor,
                   depth: torch.Tensor, estimate: torch.Tensor | None, centre_idx: int,
                   out: torch.Tensor | None = None, fallback: torch.Tensor | None = None) -> torch.Tensor:
    """One-pass assembly of the (3T-1,3,h,w) map stack (video_super_resolution.py:33-40).
    warped (T-1,h,w,3), centre (h,w,3), proj (T-1,h,w,2), resid/depth (T-1,h,w), estimate (3,h,w)|None.
    Without an estimate the last slot receives `fallback` (h,w,3): LR frame 0 of the window, as the reference's
    `else data_clone[0:1]` (:37-38); `fallback=None` keeps the centre frame there."""
    for t, n in ((warped, "warped"), (centre, "centre"), (proj, "proj"), (resid, "resid"), (depth, "depth")):
        _req(t, torch.float32, n)
    Tm1, h, w, _ = warped.shape
    T = Tm1 + 1
    if tuple(centre.shape) != (h, w, 3) or tuple(proj.shape) != (Tm1, h, w, 2) or \
            tuple(resid.shape) != (Tm1, h, w) or tuple(depth.shape) != (Tm1, h, w):
        raise ValueError("assemble_stack: inconsistent shapes")
    if estimate is not None:
        _req(estimate, torch.float32, "estimate")
        if tuple(estimate.shape) != (3, h, w):
            raise ValueError("assemble_stack: estimate must be (3,h,w)")
    if fallback is None:
        fallback = centre
    _req(fallback, torch.float32, "fallback")
    if tuple(fallback.shape) != (h, w, 3):
        raise ValueError("assemble_stack: fallback must be (h,w,3)")
    if out is None:
        out = torch.empty((3 * T - 1, 3, h, w), dtype=torch.float32, device=warped.device)
    with torch.cuda.device(warped.device):
        _lib.check(_lib.lib().vsr_assemble_stack(warped.data_ptr(), centre.data_ptr(), proj.data_ptr(), resid.data_ptr(),
                                                 depth.data_ptr(), estimate.data_ptr() if estimate is not None else None,
                                                 fallback.data_ptr(), out.data_ptr(), T, int(centre_idx), h, w, _stream()),
                   "assemble_stack")
    return out


def estimate_slot(hr: torch.Tensor, mask: torch.Tensor | None, slot: torch.Tensor, scale: int = 4) -> torch.Tensor:
    """slot (3,h,w) <- nearest-downsized hr (3,h*scale,w*scale) with masked pixels zeroed
    (video_super_resolution.py:44,58-60).  `slot` is written in place (a view of the stack)."""
    _req(hr, torch.float32, "hr")
    _req(slot, torch.float32, "slot")
    _, h, w = slot.shape
    if tuple(hr.shape) != (3, h * scale, w * scale):
        raise ValueError("estimate_slot: hr must be (3,h*scale,w*scale)")
    if mask is not None:
        _req(mask, torch.uint8, "mask")
        if tuple(mask.shape) != (h, w):
            raise ValueError("estimate_slot: mask must be (h,w)")
    with torch.cuda.device(hr.device):
        _lib.check(_lib.lib().vsr_estimate_slot(hr.data_ptr(), mask.data_ptr() if mask is not None else None,
                                                slot.data_ptr(), h, w, int(scale), _stream()), "estimate_slot")
    return slot


# -- several frame windows per launch ------------------------------------------------------------------------------
# The per-window stages above with a leading window dimension W: one launch per stage for all W windows, window b
# bit-identical to the one-window call on it (the one-window entry points are the same kernels with W = 1).

def warp_windows(frames: torch.Tensor, flows: torch.Tensor, centre: int, bilinear: bool | int = 2,
                 want_resid: bool = True):
    """warp_window over W windows: frames (W,T,H,W,3), flows (W,T-1,H,W,2) -> warped (W,T-1,H,W,3) and, with
    want_resid, resid (W,T-1,H,W)."""
    _req(frames, torch.float32, "frames")
    _req(flows, torch.float32, "flows")
    if frames.dim() != 5:
        raise ValueError("warp_windows: frames (W,T,H,W,3) expected")
    nw, T, H, W, C = frames.shape
    if nw < 1 or C != 3 or tuple(flows.shape) != (nw, T - 1, H, W, 2) or not 0 <= centre < T:
        raise ValueError("warp_windows: frames (W,T,H,W,3), flows (W,T-1,H,W,2), 0 <= centre < T expected")
    warped = torch.empty((nw, T - 1, H, W, 3), dtype=torch.float32, device=frames.device)
    resid = torch.empty((nw, T - 1, H, W), dtype=torch.float32, device=frames.device) if want_resid else None
    with torch.cuda.device(frames.device):
        _lib.check(_lib.lib().vsr_warp_windows_nhwc3(frames.data_ptr(), flows.data_ptr(), warped.data_ptr(),
                                                     resid.data_ptr() if resid is not None else None, nw, T,
                                                     int(centre), H, W, int(bilinear), _stream()), "warp_windows")
    return warped, resid


def vos_threshold_windows(logits_a: torch.Tensor, logits_b: torch.Tensor) -> torch.Tensor:
    """vos_threshold over W windows: logits (W,h,w) x2 -> mask (W,h,w) u8."""
    _req(logits_a, torch.float32, "logits_a")
    _req(logits_b, torch.float32, "logits_b")
    if logits_a.shape != logits_b.shape or logits_a.dim() != 3 or logits_a.shape[0] < 1:
        raise ValueError("vos_threshold_windows: two (W,h,w) tensors expected")
    nw, h, w = logits_a.shape
    mask = torch.empty((nw, h, w), dtype=torch.uint8, device=logits_a.device)
    with torch.cuda.device(logits_a.device):
        _lib.check(_lib.lib().vsr_vos_threshold_windows(logits_a.data_ptr(), logits_b.data_ptr(), mask.data_ptr(), nw,
                                                        h, w, _stream()), "vos_threshold_windows")
    return mask


def assemble_stacks(warped: torch.Tensor, frames: torch.Tensor, proj: torch.Tensor, resid: torch.Tensor,
                    depth: torch.Tensor, estimate: torch.Tensor | None, centre_idx: int,
                    out: torch.Tensor | None = None) -> torch.Tensor:
    """assemble_stack over W windows -> (W,3T-1,3,h,w).  warped (W,T-1,h,w,3), frames (W,T,h,w,3) (the centre frame
    and, without an estimate, the fallback LR frame 0 of each window are read from it in place), proj (W,T-1,h,w,2),
    resid / depth (W,T-1,h,w), estimate (W,3,h,w) | None."""
    for t, n in ((warped, "warped"), (frames, "frames"), (proj, "proj"), (resid, "resid"), (depth, "depth")):
        _req(t, torch.float32, n)
    if frames.dim() != 5:
        raise ValueError("assemble_stacks: frames (W,T,h,w,3) expected")
    nw, T, h, w, _ = frames.shape
    if nw < 1 or frames.shape[4] != 3 or tuple(warped.shape) != (nw, T - 1, h, w, 3) or \
            tuple(proj.shape) != (nw, T - 1, h, w, 2) or tuple(resid.shape) != (nw, T - 1, h, w) or \
            tuple(depth.shape) != (nw, T - 1, h, w) or not 0 <= centre_idx < T:
        raise ValueError("assemble_stacks: inconsistent shapes")
    if estimate is not None:
        _req(estimate, torch.float32, "estimate")
        if tuple(estimate.shape) != (nw, 3, h, w):
            raise ValueError("assemble_stacks: estimate must be (W,3,h,w)")
    if out is None:
        out = torch.empty((nw, 3 * T - 1, 3, h, w), dtype=torch.float32, device=warped.device)
    else:
        _req(out, torch.float32, "out")
        if tuple(out.shape) != (nw, 3 * T - 1, 3, h, w):
            raise ValueError("assemble_stacks: out must be (W,3T-1,3,h,w)")
    with torch.cuda.device(warped.device):
        _lib.check(_lib.lib().vsr_assemble_stack_windows(
            warped.data_ptr(), frames[0, centre_idx].data_ptr(), proj.data_ptr(), resid.data_ptr(), depth.data_ptr(),
            estimate.data_ptr() if estimate is not None else None, frames.data_ptr(), out.data_ptr(), nw,
            T * h * w * 3, T, int(centre_idx), h, w, _stream()), "assemble_stacks")
    return out


def estimate_slots(hr: torch.Tensor, mask: torch.Tensor | None, stack: torch.Tensor, scale: int = 4) -> torch.Tensor:
    """estimate_slot over W windows: the last map of each window of stack (W,M,3,h,w) <- nearest-downsized hr
    (W,3,h*scale,w*scale) with the pixels of mask (W,h,w) zeroed.  Written in place; returns stack."""
    _req(hr, torch.float32, "hr")
    _req(stack, torch.float32, "stack")
    if stack.dim() != 5 or stack.shape[2] != 3:
        raise ValueError("estimate_slots: stack must be (W,M,3,h,w)")
    nw, M, _, h, w = stack.shape
    if nw < 1 or tuple(hr.shape) != (nw, 3, h * scale, w * scale):
        raise ValueError("estimate_slots: hr must be (W,3,h*scale,w*scale)")
    if mask is not None:
        _req(mask, torch.uint8, "mask")
        if tuple(mask.shape) != (nw, h, w):
            raise ValueError("estimate_slots: mask must be (W,h,w)")
    with torch.cuda.device(hr.device):
        _lib.check(_lib.lib().vsr_estimate_slot_windows(hr.data_ptr(), mask.data_ptr() if mask is not None else None,
                                                        stack[0, M - 1].data_ptr(), nw, M * 3 * h * w, h, w,
                                                        int(scale), _stream()), "estimate_slots")
    return stack


def compose_flow_windows(g: torch.Tensor | None, f: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """compose_flow over W windows on strided views: g, f, out (W,H,W,2) with the same stride between windows (e.g.
    neighbour n of a (W,T-1,H,W,2) array, x[:, n]), each window's field contiguous.  g=None: out = f."""
    _req(f.select(0, 0), torch.float32, "f")
    for t, n in ((g, "g"), (out, "out")):
        if t is not None:
            _req(t.select(0, 0), torch.float32, n)
            if t.shape != f.shape or t.stride(0) != f.stride(0):
                raise ValueError(f"compose_flow_windows: {n} must have the shape and window stride of f")
    if f.dim() != 4 or f.shape[3] != 2 or f.shape[0] < 1:
        raise ValueError("compose_flow_windows: (W,H,W,2) fields expected")
    nw, H, W, _ = f.shape
    with torch.cuda.device(f.device):
        _lib.check(_lib.lib().vsr_compose_flow_windows(g.data_ptr() if g is not None else None, f.data_ptr(),
                                                       out.data_ptr(), nw, f.stride(0), H, W, _stream()),
                   "compose_flow_windows")
    return out


def warp_labels_windows(labels: torch.Tensor, flow: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """warp_labels over W windows: labels (W,H,W) u8, flow (W,H,W,2) with each window's field contiguous (a view such
    as x[:, n] of a (W,T-1,H,W,2) array is fine) -> (W,H,W) u8 (written into `out` when given)."""
    _req(labels, torch.uint8, "labels")
    _req(flow.select(0, 0), torch.float32, "flow")
    nw, H, W = labels.shape
    if tuple(flow.shape) != (nw, H, W, 2):
        raise ValueError("warp_labels_windows: flow must be (W,H,W,2)")
    if out is not None:
        _req(out, torch.uint8, "out")
        if out.shape != labels.shape:
            raise ValueError("warp_labels_windows: out must be (W,H,W)")
    dst = torch.empty_like(labels) if out is None else out
    with torch.cuda.device(labels.device):
        _lib.check(_lib.lib().vsr_warp_labels_u8_windows(labels.data_ptr(), flow.data_ptr(), dst.data_ptr(), nw,
                                                         flow.stride(0), H, W, _stream()), "warp_labels_windows")
    return dst


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
