"""The per-frame warp-and-fuse hot path on one GPU, and its sharding over frame windows.

`WarpFusePipeline.step` is the sequence VSR.forward runs per output frame
(network/video_super_resolution.py:23-69) with the learned estimators replaced by given geometry
(flow, inverse depth, segmentation logits -- SURVEY.md 8: FlowNet2 / MegaDepth / OSVOS bodies are
out of scope), generalised from the reference's 3-frame window to T frames (M = 3T-1 maps):

  a1  flow projection            ops.project_flow          (FlowProjectionModule)
  a2  depth-aware projection     ops.project_depth_flow    (DepthProjectionModule)
  a3  bilinear warp of the T-1 neighbour frames along the projected flow, a4 fused residual norm
  a5  mask threshold + nearest label warp                   (VOSProjectionModule)
  a7  one-pass stack assembly    ops.assemble_stack
  a6  fusion convs, pass 1       SRProjectionModule         (video_super_resolution.py:41)
  a7  downsized + masked estimate into the stack's last slot (:43-44,:57-62)
  a6  fusion convs, pass 2       SRProjectionModule         (:64)

Sharding (SURVEY.md 8e): windows are independent once the recurrence is reset at chunk starts
(main.py:196), so rank r takes a contiguous chunk of windows; no collective on the hot path.
`gather_frames` is the one collective: an all-gather of the u8-quantised output frames.
"""
from __future__ import annotations

import torch

from . import ops
from .my_packages.SRProjection.SRProjectionModule import SRProjectionModule


def shard_windows(num_windows: int, world_size: int, rank: int) -> range:
    """Contiguous chunk of window indices for `rank` (SURVEY.md 8e: [r*ceil(N/G), (r+1)*ceil(N/G)))."""
    per = -(-num_windows // world_size)
    return range(min(rank * per, num_windows), min((rank + 1) * per, num_windows))


def shard_chunks(chunks, world_size: int, rank: int) -> list:
    """Contiguous groups of whole chunks for `rank`, balanced by window count.  With the reference's own
    chunks (utils.video_utils.chunk_windows) every shard boundary is a chunk boundary, where the reference
    resets the recurrence anyway (main.py:196): the sharded result is identical to a single-GPU run."""
    chunks = [c for c in chunks if len(c) > 0]
    total = sum(len(c) for c in chunks)
    out, acc, r = [[] for _ in range(world_size)], 0, 0
    for c in chunks:
        # move on when this rank holds its share (boundaries at multiples of total / world)
        while r < world_size - 1 and acc >= (r + 1) * total / world_size:
            r += 1
        out[r].append(c)
        acc += len(c)
    return out[rank]


def shard_chunks_even(chunks, world_size: int, rank: int) -> list:
    """Even split by windows (SURVEY.md 8e: rank r takes windows [r*ceil(N/G), (r+1)*ceil(N/G))), chunks cut at the
    rank boundaries.  Better balanced than shard_chunks when there are few chunks per rank (C5: 38 windows per
    rank instead of 45/30), at the price of one extra recurrence reset where a rank boundary falls inside a
    chunk -- results differ from the single-GPU run only downstream of those resets, inside that chunk."""
    chunks = [c for c in chunks if len(c) > 0]
    total = sum(len(c) for c in chunks)
    mine = shard_windows(total, world_size, rank)
    out, base = [], 0
    for c in chunks:
        lo, hi = max(mine.start, base), min(mine.stop, base + len(c))
        if lo < hi:
            out.append(range(c.start + lo - base, c.start + hi - base))
        base += len(c)
    return out


class WarpFusePipeline:
    """Geometry (DESIGN.md 1): flows[n] is the optical flow frame n -> n+1 in frame n's coordinates.  Its projection
    (a1/a2) proj[n] lives in frame n+1's coordinates and points back to frame n.  Every neighbour is warped to the
    CENTRE frame c = T//2 with a centre -> neighbour flow G:
        past   frames t < c:  G[c-1] = proj[c-1],  G[t] = G[t+1] + proj[t](p + G[t+1])     (chain of projected flows)
        future frames t > c:  G[c+1] = flows[c],   G[t] = G[t-1] + flows[t-1](p + G[t-1])   (chain of forward flows)
    so warped[t](p) = frame[t](p + G[t](p)) is aligned with the centre frame, and the residual map of neighbour t is
    |frame[c] - warped[t]|.  The VOS mask is taken to live in frame c-1 (the frame the segmentation was propagated
    from) and is label-warped with G[c-1].  For the reference's T = 3 no chain is needed.
    max_disp: a promised bound on the components of `flows` (px); selects the shared-memory projection path.
    reuse: what the fuse pass (pass 2) takes over from pass 1.  The M maps go through the conv stack independently
    until the per-pixel fc, so a map that enters both passes unchanged need not be convolved twice (bit-identical):
        None         every map again (the default: the reference's two full SRProjectionModule calls)
        "frames"     the T frame maps, which network/video_super_resolution.py:62 feeds unchanged (`data`), are reused;
                     the 2(T-1) flow / depth maps, which the reference re-estimates for pass 2, and the estimate are not
        "unchanged"  every map this pipeline leaves unchanged: all but the estimate slot (flow and depth are inputs
                     here, not re-estimated)."""

    def __init__(self, T: int, h: int, w: int, sr: SRProjectionModule | None = None, scale: int = 4,
                 device="cuda:0", run_fusion: bool = True, max_disp: float | None = None, reuse: str | None = None):
        if T < 2:
            raise ValueError("window must hold at least 2 frames")
        if reuse not in (None, "frames", "unchanged"):
            raise ValueError("reuse must be None, 'frames' or 'unchanged'")
        self.reuse = reuse
        self.T, self.h, self.w, self.scale = T, h, w, scale
        self.M = 3 * T - 1
        self.centre = T // 2
        self.device = torch.device(device)
        self.run_fusion = run_fusion
        self.max_disp = max_disp
        self.sr = sr if sr is not None else SRProjectionModule(num_maps=self.M)
        if self.sr.num_maps != self.M:
            raise ValueError(f"SRProjectionModule.num_maps={self.sr.num_maps}, window needs {self.M}")
        self.stack = torch.empty((self.M, 3, h, w), dtype=torch.float32, device=self.device)
        self.centre_flows = torch.empty((T - 1, h, w, 2), dtype=torch.float32, device=self.device)

    def chain_flows(self, proj, flows):
        """Fills self.centre_flows (T-1,h,w,2): neighbour order = frame order with the centre left out."""
        T, c, G = self.T, self.centre, self.centre_flows
        ops.compose_flow(None, proj[c - 1], out=G[c - 1])
        for t in range(c - 2, -1, -1):
            ops.compose_flow(G[t + 1], proj[t], out=G[t])
        if c + 1 < T:
            ops.compose_flow(None, flows[c], out=G[c])               # frame c+1 is neighbour index c
            for t in range(c + 2, T):
                ops.compose_flow(G[t - 2], flows[t - 1], out=G[t - 1])
        return G

    def project_and_warp(self, frames, flows, inv_depth, logits_a, logits_b, estimate=None, estimate_hr=None):
        """a1-a5 + a7: fills self.stack; returns the intermediate results (for tests).
        estimate: (3,h,w) LR estimate | None; estimate_hr: (3,s*h,s*w) the previous output frame, downsized here
        (video_super_resolution.py:35-37); neither: LR frame 0 (:38)."""
        T, c = self.T, self.centre
        proj_f, _, cnt_f, hole_f = ops.project_flow(flows, None, self.max_disp)
        proj_d, wsum, cnt_d, hole_d = ops.project_depth_flow(flows, inv_depth, self.max_disp)
        G = self.chain_flows(proj_d, flows)
        warped, resid = ops.warp_window(frames, G, c, 2)          # fast fp32 blend (north star: <= 1e-3)
        mask = ops.vos_threshold(logits_a, logits_b)
        mask_w = ops.warp_labels(mask.unsqueeze(0), G[c - 1].unsqueeze(0))[0]
        ops.assemble_stack(warped, frames[c], proj_f, resid, wsum, estimate, c, out=self.stack, fallback=frames[0])
        if estimate is None and estimate_hr is not None:
            ops.estimate_slot(estimate_hr, None, self.stack[self.M - 1], self.scale)
        return {"proj_flow": proj_f, "count_flow": cnt_f, "hole_flow": hole_f, "proj_depth": proj_d, "wsum": wsum,
                "count_depth": cnt_d, "hole_depth": hole_d, "warped": warped, "resid": resid, "mask": mask,
                "mask_warped": mask_w, "centre_flows": G}

    def step(self, frames, flows, inv_depth, logits_a, logits_b, estimate=None, estimate_hr=None, out_u8=None,
             want_f32=True):
        """frames (T,h,w,3) 0..255, flows (T-1,h,w,2), inv_depth (T-1,h,w), logits (h,w) x2,
        estimate (3,h,w)|None -> SR frame (1,3,s*h,s*w) fp32 [and / or out_u8 (s*h,s*w,3) u8].
        Every kernel between the first and the last launch of a step is this library's."""
        r = self.project_and_warp(frames, flows, inv_depth, logits_a, logits_b, estimate, estimate_hr)
        if not self.run_fusion:
            return self.stack
        out1 = self.sr(self.stack)                                             # pass 1
        ops.estimate_slot(out1[0], r["mask_warped"], self.stack[self.M - 1], self.scale)
        changed_from = {None: None, "frames": self.T, "unchanged": self.M - 1}[self.reuse]
        return self.sr(self.stack, out_u8=out_u8, want_f32=want_f32, changed_from=changed_from)   # pass 2 (fuse)


class GraphedStep:
    """The per-frame sequence of WarpFusePipeline.step captured once into a CUDA graph (SURVEY.md 7 step 6) and replayed:
    ~190 launches (projection stages, flow chains, warps, stack, two conv-stack passes) become one graph launch.
    Inputs live in static device buffers (`inputs`: copy -- or H2D-copy -- each window into them, then `replay()`);
    outputs are the static `frame_u8` (s*h, s*w, 3) and, with want_f32, `frame` (1,3,s*h,s*w).
    The step is GPU-bound (100 ms of kernels against ~1 ms of launch calls), so this buys little at C2; it matters for
    small frames, where the front's 40 launches of 5-10 us each are launch-latency bound.
    The graph holds whichever projection path torch.are_deterministic_algorithms_enabled() selected at capture time
    (ops.project_flow): changing the flag afterwards does not change what replay() runs."""

    def __init__(self, pipe: "WarpFusePipeline", want_f32: bool = False, warmup: int = 2):
        T, h, w, s, dev = pipe.T, pipe.h, pipe.w, pipe.scale, pipe.device
        f32 = dict(dtype=torch.float32, device=dev)
        self.pipe = pipe
        self.inputs = {"frames": torch.zeros((T, h, w, 3), **f32), "flows": torch.zeros((T - 1, h, w, 2), **f32),
                       "inv_depth": torch.ones((T - 1, h, w), **f32), "logits_a": torch.zeros((h, w), **f32),
                       "logits_b": torch.zeros((h, w), **f32)}
        self.frame_u8 = torch.empty((s * h, s * w, 3), dtype=torch.uint8, device=dev)
        self.frame = None
        i = self.inputs
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):          # warm-up on the capture stream: plans, function attributes, workspaces
            for _ in range(max(warmup, 1)):
                pipe.step(i["frames"], i["flows"], i["inv_depth"], i["logits_a"], i["logits_b"], out_u8=self.frame_u8,
                          want_f32=want_f32)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            y = pipe.step(i["frames"], i["flows"], i["inv_depth"], i["logits_a"], i["logits_b"], out_u8=self.frame_u8,
                          want_f32=want_f32)
        if want_f32:
            self.frame = y

    def load(self, frames, flows, inv_depth, logits_a, logits_b, non_blocking=True):
        for k, v in zip(("frames", "flows", "inv_depth", "logits_a", "logits_b"), (frames, flows, inv_depth, logits_a, logits_b)):
            self.inputs[k].copy_(v, non_blocking=non_blocking)

    def replay(self):
        self.graph.replay()
        return self.frame if self.frame is not None else self.frame_u8


def quantise_u8(frame: torch.Tensor) -> torch.Tensor:
    """(1,3,H,W) fp32 0..255 -> (H,W,3) u8, the format the reference's loader reads (utils/video_utils.py:23)."""
    return frame[0].clamp(0, 255).round().to(torch.uint8).permute(1, 2, 0).contiguous()


def gather_frames(local_frames: torch.Tensor, group=None) -> torch.Tensor:
    """All-gather of each rank's (n,H,W,3) u8 output frames into (world*n,H,W,3), rank-major = window
    order under shard_windows.  The only collective of the pipeline (NCCL over NVLink on GPUs, gloo in
    the CPU tests)."""
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return local_frames
    world = dist.get_world_size(group)
    out = torch.empty((world,) + tuple(local_frames.shape), dtype=local_frames.dtype, device=local_frames.device)
    if local_frames.is_cuda:
        dist.all_gather_into_tensor(out, local_frames.contiguous(), group=group)      # ncclAllGather
    else:
        dist.all_gather(list(out.unbind(0)), local_frames.contiguous(), group=group)  # gloo (CPU tests)
    return out.flatten(0, 1)


def gather_frames_ragged(local_frames: torch.Tensor, group=None) -> torch.Tensor:
    """gather_frames for shards of unequal length: counts are exchanged first, shards are padded to the
    longest one for the single all-gather, and the padding is dropped."""
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return local_frames
    world = dist.get_world_size(group)
    n = torch.tensor([local_frames.shape[0]], dtype=torch.int64, device=local_frames.device)
    counts = torch.zeros(world, dtype=torch.int64, device=local_frames.device)
    if local_frames.is_cuda:
        dist.all_gather_into_tensor(counts, n, group=group)
    else:
        dist.all_gather(list(counts.unbind(0)), n[0], group=group)
    counts = counts.tolist()
    m = max(counts)
    pad = torch.zeros((m,) + tuple(local_frames.shape[1:]), dtype=local_frames.dtype, device=local_frames.device)
    pad[:local_frames.shape[0]] = local_frames
    allf = gather_frames(pad, group).unflatten(0, (world, m))
    return torch.cat([allf[r, :counts[r]] for r in range(world)])


def run_sequence(vsr, frames, flows, inv_depth, logits, chunks, out: torch.Tensor | None = None):
    """The reference's loop over a video (main.py:190-203) on this rank's chunks.

    frames (N,h,w,3) fp32 0..255, flows (N-1,h,w,2), inv_depth (N-1,h,w) on the device; logits: callable
    k -> (logits_a, logits_b) for window k; chunks: list of ranges of window indices (shard_chunks).
    Within a chunk window k+1 receives window k's output as its estimate; every chunk starts with
    estimated_image = None.  Returns (u8 frames (n_local,H,W,3), list of window indices)."""
    T = vsr.window
    idx = [k for c in chunks for k in c]
    s = vsr.model.upscale_factor
    h, w = frames.shape[1:3]
    if out is None:
        out = torch.empty((len(idx), s * h, s * w, 3), dtype=torch.uint8, device=frames.device)
    pipe = vsr._pipe(h, w, frames.device)
    i = 0
    for c in chunks:
        est = None                                                   # recurrence reset at every chunk start (main.py:196)
        for k in c:
            la, lb = logits(k)
            # the previous output frame stays planar fp32 on the device and is downsized into the estimate slot by
            # vsr_estimate_slot; the u8 frame (utils/video_utils.py:23) is written by the fc-fuse kernel itself
            est = pipe.step(frames[k:k + T], flows[k:k + T - 1], inv_depth[k:k + T - 1], la, lb,
                            estimate_hr=None if est is None else est[0], out_u8=out[i])
            i += 1
    return out, idx
