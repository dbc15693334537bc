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
Window batching: `WarpFusePipeline(..., windows=W)` runs W independent windows per step with one launch per stage,
and `run_sequence(..., windows=W)` uses it to advance W of a rank's chunks in lockstep.
`gather_frames` is the one collective: an all-gather of the u8-quantised output frames.
Map groups (DESIGN.md 11): `WarpFusePipeline(..., map_group=pg)` runs ONE window over the G GPUs of an NCCL group --
rank 0 builds the stack and broadcasts it, each rank convolves its share of the maps and fuses its row band -- with
frames bit-identical to one GPU, so `run_sequence(..., map_group=pg)` runs one recurrence on G GPUs.
"""
from __future__ import annotations

import torch

from . import ops
from .map_parallel import as_map_group
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
                     here, not re-estimated).
    windows: W independent frame windows per step (default 1).  Every stage is one launch for all W windows and window
    b's results are bit-identical to a one-window step on it.  With W > 1 the inputs and outputs carry a leading window
    dimension: frames (W,T,h,w,3), flows (W,T-1,h,w,2), inv_depth (W,T-1,h,w), logits (W,h,w), estimate (W,3,h,w),
    estimate_hr (W,3,s*h,s*w); the stack is (W,M,3,h,w) and the SR frames (W,3,s*h,s*w).  With W = 1 the one-window
    shapes are taken as before (and the batched ones with a leading 1).
    map_group: an NCCL process group of G ranks (one GPU each) that runs each step together, one window (windows must
    be 1).  Rank 0 builds the stack and VOS mask (a1-a5, a7) and broadcasts them -- with the default atomic projection
    their fp32 sums can differ in the last bits from rank to rank, and the frame must be fused from maps of ONE stack;
    the ranks then split the conv stack by maps and the fc by row bands (SRProjectionModule(map_group=...), which `sr`
    must be, with the same group).  The estimate slot is written band by band (vsr_estimate_slot_windows on each rank's
    rows) and all-gathered.  Every rank passes the same inputs; rank 0's are the ones used."""

    def __init__(self, T: int, h: int, w: int, sr: SRProjectionModule | None = None, scale: int = 4,
                 device="cuda:0", run_fusion: bool = True, max_disp: float | None = None, reuse: str | None = None,
                 windows: int = 1, map_group=None):
        if T < 2:
            raise ValueError("window must hold at least 2 frames")
        if reuse not in (None, "frames", "unchanged"):
            raise ValueError("reuse must be None, 'frames' or 'unchanged'")
        if int(windows) != windows or windows < 1:
            raise ValueError("windows must be an integer >= 1")
        self.reuse = reuse
        self.T, self.h, self.w, self.scale = T, h, w, scale
        self.windows = W = int(windows)
        self.M = 3 * T - 1
        self._changed_from = {None: None, "frames": T, "unchanged": self.M - 1}[reuse]   # pass 2 convolves maps >= it
        self.centre = T // 2
        self.device = torch.device(device)
        self.run_fusion = run_fusion
        self.max_disp = max_disp
        self.map_group = mg = as_map_group(map_group)
        if mg is not None and W > 1:
            raise ValueError("WarpFusePipeline: windows > 1 is not supported with a map group")
        if sr is not None and getattr(sr.map_group, "pg", sr.map_group) is not getattr(mg, "pg", mg):
            raise ValueError("WarpFusePipeline: sr must be an SRProjectionModule built with the same map_group")
        self.sr = sr if sr is not None else SRProjectionModule(num_maps=self.M, map_group=mg)
        if self.sr.num_maps != self.M:
            raise ValueError(f"SRProjectionModule.num_maps={self.sr.num_maps}, window needs {self.M}")
        lead = (W,) if W > 1 else ()
        if mg is None:
            self.stack = torch.empty(lead + (self.M, 3, h, w), dtype=torch.float32, device=self.device)
            self._mask_w = torch.empty((W, h, w), dtype=torch.uint8, device=self.device)
        else:
            self.map_group = mg = self.sr.map_group
            (_, _), lb, _ = self.sr.band_geometry(h)        # ValueError for fewer LR rows than ranks
            # stack and warped VOS mask in one buffer: one broadcast from rank 0
            nst = self.M * 3 * h * w
            self._bcast = torch.empty(nst * 4 + h * w, dtype=torch.uint8, device=self.device)
            self.stack = self._bcast[:nst * 4].view(torch.float32).view(self.M, 3, h, w)
            self._mask_w = self._bcast[nst * 4:].view(1, h, w)
            hmax = max(lb[p + 1] - lb[p] for p in range(mg.size))
            self._slot_send = torch.empty(3 * hmax * w, dtype=torch.float32, device=self.device)
            self._slot_all = torch.empty(mg.size * 3 * hmax * w, dtype=torch.float32, device=self.device)
        self.centre_flows = torch.empty(lead + (T - 1, h, w, 2), dtype=torch.float32, device=self.device)
        self._stack = self.stack.view(W, self.M, 3, h, w)          # window-major views of the same storage
        self._centre_flows = self.centre_flows.view(W, T - 1, h, w, 2)

    def chain_flows(self, proj, flows):
        """Fills self.centre_flows ([W,]T-1,h,w,2): neighbour order = frame order with the centre left out.
        proj / flows: ([W,]T-1,h,w,2).  One launch per link for all windows."""
        T, c, G, W = self.T, self.centre, self._centre_flows, self.windows
        proj = proj.reshape(W, T - 1, self.h, self.w, 2)
        flows = flows.reshape(W, T - 1, self.h, self.w, 2)
        ops.compose_flow(None, proj[:, c - 1], out=G[:, c - 1])
        for t in range(c - 2, -1, -1):
            ops.compose_flow(G[:, t + 1], proj[:, t], out=G[:, t])
        if c + 1 < T:
            ops.compose_flow(None, flows[:, c], out=G[:, c])     # frame c+1 is neighbour index c
            for t in range(c + 2, T):
                ops.compose_flow(G[:, t - 2], flows[:, t - 1], out=G[:, t - 1])
        return self.centre_flows

    def _batched(self, frames, flows, inv_depth, logits_a, logits_b, estimate, estimate_hr):
        """The inputs as window-major (W,...) tensors; raises ValueError on a shape that fits neither form."""
        W, T, h, w, s = self.windows, self.T, self.h, self.w, self.scale
        single = W == 1 and frames.dim() == 4
        lead = () if single else (W,)
        want = {"frames": (T, h, w, 3), "flows": (T - 1, h, w, 2), "inv_depth": (T - 1, h, w), "logits_a": (h, w),
                "logits_b": (h, w), "estimate": (3, h, w), "estimate_hr": (3, s * h, s * w)}
        got = {"frames": frames, "flows": flows, "inv_depth": inv_depth, "logits_a": logits_a, "logits_b": logits_b,
               "estimate": estimate, "estimate_hr": estimate_hr}
        for k, t in got.items():
            if t is not None and tuple(t.shape) != lead + want[k]:
                raise ValueError(f"WarpFusePipeline: {k} must be {lead + want[k]}, got {tuple(t.shape)}")
            if t is not None and not t.is_contiguous():
                raise ValueError(f"WarpFusePipeline: {k}: tensor must be contiguous")
        return {k: (t.unsqueeze(0) if single and t is not None else t) for k, t in got.items()}, single

    def project_and_warp(self, frames, flows, inv_depth, logits_a, logits_b, estimate=None, estimate_hr=None,
                         estimate_hr_windows=None):
        """a1-a5 + a7: fills self.stack; returns the intermediate results (for tests), with the leading window
        dimension when the inputs have it.
        estimate: ([W,]3,h,w) LR estimate | None; estimate_hr: ([W,]3,s*h,s*w) the previous output frame, downsized here
        (video_super_resolution.py:35-37); neither: LR frame 0 (:38).  estimate_hr_windows: the windows that take
        estimate_hr (default all); the others keep LR frame 0."""
        x, single = self._batched(frames, flows, inv_depth, logits_a, logits_b, estimate, estimate_hr)
        W, T, c, h, w = self.windows, self.T, self.centre, self.h, self.w
        fl = x["flows"].reshape(W * (T - 1), h, w, 2)
        proj_f, _, cnt_f, hole_f = ops.project_flow(fl, None, self.max_disp)
        proj_d, wsum, cnt_d, hole_d = ops.project_depth_flow(fl, x["inv_depth"].reshape(W * (T - 1), h, w),
                                                             self.max_disp)
        self.chain_flows(proj_d, fl)
        G = self._centre_flows
        warped, resid = ops.warp_window(x["frames"], G, c, 2)      # fast fp32 blend (north star: <= 1e-3)
        mask = ops.vos_threshold(x["logits_a"], x["logits_b"])
        mask_w = ops.warp_labels(mask, G[:, c - 1], out=self._mask_w)
        ops.assemble_stack(warped, x["frames"], proj_f.view(W, T - 1, h, w, 2), resid, wsum.view(W, T - 1, h, w),
                           x["estimate"], c, out=self._stack)
        if estimate is None and estimate_hr is not None:
            sel = range(W) if estimate_hr_windows is None else sorted(set(estimate_hr_windows))
            for a, b in _runs(sel):                                    # one launch per run of consecutive windows
                ops.estimate_slot(x["estimate_hr"][a:b], None, self._stack[a:b, self.M - 1], self.scale)
        r = {"proj_flow": proj_f, "count_flow": cnt_f, "hole_flow": hole_f, "proj_depth": proj_d, "wsum": wsum,
             "count_depth": cnt_d, "hole_depth": hole_d}
        r = {k: v.view((W, T - 1) + tuple(v.shape[1:])) for k, v in r.items()}
        r.update({"warped": warped, "resid": resid, "mask": mask, "mask_warped": mask_w, "centre_flows": G})
        return {k: v[0] for k, v in r.items()} if single else r

    def step(self, frames, flows, inv_depth, logits_a, logits_b, estimate=None, estimate_hr=None, out_u8=None,
             want_f32=True, estimate_hr_windows=None, estimate_hr_band=None, gather=True):
        """frames (T,h,w,3) 0..255, flows (T-1,h,w,2), inv_depth (T-1,h,w), logits (h,w) x2,
        estimate (3,h,w)|None -> SR frame (1,3,s*h,s*w) fp32 [and / or out_u8 (s*h,s*w,3) u8].
        With W windows: the same with a leading W (class docstring) -> (W,3,s*h,s*w) [and / or out_u8 (W,s*h,s*w,3)].
        With a map group: estimate_hr_band = this rank's row band (1,3,rows,s*w) of the previous output frame (what a step
        with gather="u8" or False returns), the recurrence without a gathered fp32 frame; `gather` as
        SRProjectionModule.forward (True: full frames on every rank; "u8": out_u8 gathered, this rank's fp32 band
        returned; False: this rank's band only).
        Every kernel between the first and the last launch of a step is this library's (and, with a map group, NCCL's)."""
        mg = self.map_group
        if mg is None and (estimate_hr_band is not None or gather is not True):
            raise ValueError("WarpFusePipeline: estimate_hr_band and gather need a map group")
        if mg is None or mg.rank == 0:
            self.project_and_warp(frames, flows, inv_depth, logits_a, logits_b, estimate, estimate_hr,
                                  estimate_hr_windows)
        if mg is not None:
            mg.broadcast(self._bcast, 0)                   # the stack and mask every rank convolves
        if not self.run_fusion:
            return self.stack
        if mg is None:
            ops.estimate_slot(self.sr(self.stack), self._mask_w, self._stack[:, self.M - 1], self.scale)   # pass 1
        else:
            if estimate_hr_band is not None:
                self._slot_from_band(estimate_hr_band, None)
            self._slot_from_band(self.sr(self.stack, gather=False), self._mask_w[0])    # pass 1: this rank's band
        return self.sr(self.stack, out_u8=out_u8, want_f32=want_f32, changed_from=self._changed_from,   # pass 2 (fuse)
                       gather=gather)

    def _slot_from_band(self, band, mask):
        """The estimate slot from the frame's row bands: each rank downsizes its band into its LR rows of the slot
        (vsr_estimate_slot_windows with the band as the frame), and an all-gather assembles the (3,h,w) slot on every
        rank."""
        mg, s, w = self.map_group, self.scale, self.w
        _, lb, hb = self.sr.band_geometry(self.h)
        r = mg.rank
        rows, lrows = hb[r + 1] - hb[r], lb[r + 1] - lb[r]
        if band.numel() != 3 * rows * s * w:
            raise ValueError(f"WarpFusePipeline: estimate band must be (1,3,{rows},{s * w}), got {tuple(band.shape)}")
        slot = self._slot_send[:3 * lrows * w].view(3, lrows, w)
        ops.estimate_slot(band.reshape(3, rows, s * w), None if mask is None else mask[lb[r]:lb[r + 1]], slot, s)
        mg.all_gather(self._slot_all, self._slot_send)
        ops.unpack_bands(self._slot_all, self.stack[self.M - 1], lb, 3, w, self._slot_send.numel())


def _runs(sel):
    """[a, b) ranges of consecutive integers in the sorted sequence sel."""
    out = []
    for k in sel:
        if out and out[-1][1] == k:
            out[-1][1] = k + 1
        else:
            out.append([k, k + 1])
    return [tuple(r) for r in out]


class GraphedStep:
    """The per-frame sequence of WarpFusePipeline.step captured once into a CUDA graph (SURVEY.md 7 step 6) and replayed:
    ~190 launches (projection stages, flow chains, warps, stack, two conv-stack passes) become one graph launch.
    Inputs live in static device buffers (`inputs`: copy -- or H2D-copy -- each window into them, then `replay()`);
    outputs are the static `frame_u8` (s*h, s*w, 3) and, with want_f32, `frame` (1,3,s*h,s*w); for a pipeline of W > 1
    windows the inputs and `frame_u8` have a leading W and `frame` is (W,3,s*h,s*w).
    The step is GPU-bound (100 ms of kernels against ~1 ms of launch calls), so this buys little at C2; it matters for
    small frames, where the front's 40 launches of 5-10 us each are launch-latency bound.
    The graph holds whichever projection path torch.are_deterministic_algorithms_enabled() selected at capture time
    (ops.project_flow): changing the flag afterwards does not change what replay() runs."""

    def __init__(self, pipe: "WarpFusePipeline", want_f32: bool = False, warmup: int = 2):
        T, h, w, s, dev = pipe.T, pipe.h, pipe.w, pipe.scale, pipe.device
        f32 = dict(dtype=torch.float32, device=dev)
        self.pipe = pipe
        n = (pipe.windows,) if pipe.windows > 1 else ()       # a W-window pipeline: every buffer has a leading W
        self.inputs = {"frames": torch.zeros(n + (T, h, w, 3), **f32), "flows": torch.zeros(n + (T - 1, h, w, 2), **f32),
                       "inv_depth": torch.ones(n + (T - 1, h, w), **f32), "logits_a": torch.zeros(n + (h, w), **f32),
                       "logits_b": torch.zeros(n + (h, w), **f32)}
        self.frame_u8 = torch.empty(n + (s * h, s * w, 3), dtype=torch.uint8, device=dev)
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


def run_sequence(vsr, frames, flows, inv_depth, logits, chunks, out: torch.Tensor | None = None, windows: int = 1,
                 map_group=None):
    """The reference's loop over a video (main.py:190-203) on this rank's chunks.

    frames (N,h,w,3) fp32 0..255, flows (N-1,h,w,2), inv_depth (N-1,h,w) on the device; logits: callable
    k -> (logits_a, logits_b) for window k; chunks: list of ranges of window indices (shard_chunks).
    Within a chunk window k+1 receives window k's output as its estimate; every chunk starts with
    estimated_image = None.  Returns (u8 frames (n_local,H,W,3), list of window indices).
    windows=W > 1: up to W chunks advance in lockstep, one window of each per step of a W-window pipeline
    (WarpFusePipeline(windows=W)), each with its own recurrence; a slot whose chunk ends takes the next chunk.  The
    frames, and their order, are those of the one-window loop.
    map_group=pg: one recurrence on the G GPUs of the group (vsr = VSR(..., map_group=pg)); every rank of the group
    calls this with the same chunks and receives the same u8 frames, bit-identical to the one-GPU loop.  Each step
    passes only this rank's fp32 row band of its output on as the next estimate.  With a world of groups x G ranks
    (map_parallel.new_map_groups) each group runs its shard_chunks(chunks, num_groups, group index)."""
    if int(windows) != windows or windows < 1:
        raise ValueError("windows must be an integer >= 1")
    if map_group is not None:
        own = vsr.model.map_group
        if own is None or getattr(own, "pg", own) is not getattr(map_group, "pg", map_group):
            raise ValueError("run_sequence: map_group must be the group the VSR was built with (VSR(map_group=...))")
        if windows > 1:
            raise ValueError("run_sequence: windows > 1 is not supported with a map group")
    if windows > 1:
        return _run_lockstep(vsr, frames, flows, inv_depth, logits, chunks, out, int(windows))
    T = vsr.window
    idx = [k for c in chunks for k in c]
    s = vsr.model.upscale_factor
    h, w = frames.shape[1:3]
    if out is None:
        out = torch.empty((len(idx), s * h, s * w, 3), dtype=torch.uint8, device=frames.device)
    pipe = vsr._pipe(h, w, frames.device)
    group = pipe.map_group is not None
    i = 0
    for c in chunks:
        est = None                                                   # recurrence reset at every chunk start (main.py:196)
        for k in c:
            la, lb = logits(k)
            # the previous output frame stays planar fp32 on the device and is downsized into the estimate slot by
            # vsr_estimate_slot_windows (a map group keeps only this rank's row band of it and all-gathers the u8
            # frame); the u8 frame (utils/video_utils.py:23) is written by the fc-fuse kernel itself
            if group:
                nxt = {"estimate_hr_band": est, "gather": "u8"}
            else:
                nxt = {"estimate_hr": None if est is None else est[0]}
            est = pipe.step(frames[k:k + T], flows[k:k + T - 1], inv_depth[k:k + T - 1], la, lb, out_u8=out[i], **nxt)
            i += 1
    return out, idx


def _run_lockstep(vsr, frames, flows, inv_depth, logits, chunks, out, W):
    """run_sequence with W chunk slots.  Each step gathers one window per slot into the pipeline's (W,...) inputs (device
    copies), runs one batched step and copies the live slots' u8 frames to their places in `out`.  Slot j's estimate
    is frame j of the previous step's fp32 output unless its chunk just started (then LR frame 0, as the one-window
    loop).  A slot without a chunk left (the tail) repeats a live slot's inputs and its frame is dropped."""
    T = vsr.window
    chunks = [c for c in chunks if len(c) > 0]
    idx = [k for c in chunks for k in c]
    s = vsr.model.upscale_factor
    h, w = frames.shape[1:3]
    dev = frames.device
    if out is None:
        out = torch.empty((len(idx), s * h, s * w, 3), dtype=torch.uint8, device=dev)
    if not chunks:
        return out, idx
    pipe = vsr._pipe(h, w, dev, windows=W)
    f32 = dict(dtype=torch.float32, device=dev)
    fb, flb = torch.empty((W, T, h, w, 3), **f32), torch.empty((W, T - 1, h, w, 2), **f32)
    db, lab, lbb = torch.empty((W, T - 1, h, w), **f32), torch.empty((W, h, w), **f32), torch.empty((W, h, w), **f32)
    ub = torch.empty((W, s * h, s * w, 3), dtype=torch.uint8, device=dev)
    starts, acc = [], 0                                  # position of each chunk's first frame in `out`
    for c in chunks:
        starts.append(acc)
        acc += len(c)
    nxt = 0
    slots = []                                           # per slot: [chunk number, position in the chunk] or None
    for _ in range(W):
        slots.append([nxt, 0] if nxt < len(chunks) else None)
        nxt += 1 if nxt < len(chunks) else 0
    prev = None
    while any(sl is not None for sl in slots):
        live = [j for j, sl in enumerate(slots) if sl is not None]
        for j in range(W):
            ci, pos = slots[j] if slots[j] is not None else slots[live[0]]
            k = chunks[ci][pos]
            fb[j].copy_(frames[k:k + T])
            flb[j].copy_(flows[k:k + T - 1])
            db[j].copy_(inv_depth[k:k + T - 1])
            la, lb = logits(k)
            lab[j].copy_(la)
            lbb[j].copy_(lb)
        est = [j for j in live if slots[j][1] > 0]
        prev = pipe.step(fb, flb, db, lab, lbb, estimate_hr=prev if est else None, estimate_hr_windows=est, out_u8=ub)
        for j in live:
            ci, pos = slots[j]
            out[starts[ci] + pos].copy_(ub[j])
            if pos + 1 < len(chunks[ci]):
                slots[j][1] = pos + 1
            elif nxt < len(chunks):
                slots[j] = [nxt, 0]                      # the next chunk starts in this slot: recurrence reset
                nxt += 1
            else:
                slots[j] = None
    return out, idx
