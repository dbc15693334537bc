"""Helpers shared by the front's GPU tests: a warp through the C ABI into an output carved at a chosen offset of a
larger buffer (ops.warp always allocates a 16-byte-aligned output, so its unaligned store paths are reachable only
this way), and the poisoning of the projection workspace."""
import torch

from video_super_resolution_b200 import _lib, ops


def warp_carved(src, flow, mode, ref=None, offset_floats=1):
    """vsr_warp_nhwc_f32 of src (B,H,W,C) by flow (B,H,W,2) into a (B,H,W,C) view that starts offset_floats floats into
    its buffer (offset 1: 4 bytes past a 16-byte boundary, so the C = 3 kernel takes its scalar stores).  Returns
    (warped, norm), norm None without ref."""
    B, H, W, C = src.shape
    buf = torch.empty(src.numel() + offset_floats, dtype=torch.float32, device=src.device)
    dst = buf[offset_floats:].view(B, H, W, C)
    assert dst.data_ptr() % 16 == 4 * (offset_floats % 4)
    norm = torch.empty((B, H, W), dtype=torch.float32, device=src.device) if ref is not None else None
    with torch.cuda.device(src.device):
        _lib.check(_lib.lib().vsr_warp_nhwc_f32(src.data_ptr(), flow.data_ptr(), dst.data_ptr(),
                                                ref.data_ptr() if ref is not None else None,
                                                norm.data_ptr() if norm is not None else None, B, H, W, C, int(mode),
                                                torch.cuda.current_stream().cuda_stream), "warp")
    return dst, norm


def poison_workspaces():
    """The projection workspace may hold anything (include/vsr_b200.h): fill every cached one with 0xA5 bytes, so that
    a path which leaves part of it unwritten cannot be rescued by what an earlier call left there."""
    for ws in ops._WORKSPACES.values():
        ws.fill_(0xA5)
