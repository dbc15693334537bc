"""GPU: one frame window over a map group (DESIGN.md 11).  Every frame must be bit-identical (torch.equal) to the one-GPU
result: the SR stack alone (fp32 and u8, x4 and x2, bands of unequal height, M = 8 and 20, a workspace cap that chunks
inside a rank's map range, changed_from), the pipeline step (every reuse mode, the banded estimate of the next step),
run_sequence over two chunks, and groups x G chunk sharding.

Each case runs once per rank and compares that rank's results with the one-GPU path computed on its own device.  It
runs twice over:
  * G ranks as threads on one device, with `_ThreadRank` standing in for the NCCL group (the same four collectives,
    as device copies; the all_to_all checks that every rank's split sizes match its peers');
  * G NCCL ranks on G devices (torch.multiprocessing.spawn), skipped when there are fewer devices -- G = 1 runs the
    real collectives on one device.
"""
import os
import socket
import threading

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import srfbn_oracle as so
from video_super_resolution_b200 import ops, synthetic as syn
from video_super_resolution_b200.map_parallel import MapGroup, map_ranges, new_map_groups
from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
from video_super_resolution_b200.network.video_super_resolution import VSR
from video_super_resolution_b200.pipeline import WarpFusePipeline, run_sequence, shard_chunks
from video_super_resolution_b200.utils.video_utils import chunk_windows

pytestmark = pytest.mark.gpu


# -- G ranks as threads on one device ---------------------------------------------------------------------------------
class _Hub:
    def __init__(self, G):
        self.barrier = threading.Barrier(G, timeout=600)
        self.slots = [None] * G


class _ThreadRank:
    """MapGroup stand-in for rank `rank` of G threads sharing one device."""

    def __init__(self, hub, rank, size):
        self.hub, self.rank, self.size = hub, rank, size

    def _publish(self, item):
        torch.cuda.current_stream().synchronize()
        self.hub.slots[self.rank] = item
        self.hub.barrier.wait()
        return list(self.hub.slots)

    def _done(self):
        torch.cuda.current_stream().synchronize()
        self.hub.barrier.wait()                 # nobody republishes before every rank has read

    def broadcast(self, t, src=0):
        slots = self._publish(t)
        if self.rank != src:
            t.copy_(slots[src])
        self._done()

    def all_to_all(self, out, inp, out_splits, in_splits):
        assert sum(in_splits) == inp.numel() and sum(out_splits) == out.numel()
        slots = self._publish((inp, list(in_splits)))
        o = 0
        for q in range(self.size):
            qi, qs = slots[q]
            assert qs[self.rank] == out_splits[q], (q, self.rank, qs, out_splits)
            a = sum(qs[:self.rank])
            out[o:o + out_splits[q]].copy_(qi[a:a + out_splits[q]])
            o += out_splits[q]
        self._done()

    def all_gather(self, out, inp):
        slots = self._publish(inp)
        n = inp.numel()
        assert out.numel() == self.size * n
        for q in range(self.size):
            assert slots[q].numel() == n
            out[q * n:(q + 1) * n].copy_(slots[q])
        self._done()


def _threads(G, case, *args):
    hub, res, errs = _Hub(G), [None] * G, []

    def body(r):
        try:
            with torch.cuda.stream(torch.cuda.Stream("cuda:0")):
                res[r] = case(_ThreadRank(hub, r, G), torch.device("cuda:0"), *args)
                torch.cuda.current_stream().synchronize()
        except BaseException as e:           # noqa: BLE001 -- reported below; the other ranks must not wait for it
            errs.append(e)
            hub.barrier.abort()

    ts = [threading.Thread(target=body, args=(r,)) for r in range(G)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    if errs:
        raise errs[0]
    return res


# -- G NCCL ranks, one device each ------------------------------------------------------------------------------------
def _nccl_worker(rank, G, port, name, args, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=G, device_id=dev)
    try:
        torch.use_deterministic_algorithms(True)
        out[rank] = CASES[name](MapGroup(dist.group.WORLD), dev, *args)
    finally:
        dist.destroy_process_group()


def _nccl(G, name, *args):
    if torch.cuda.device_count() < G:
        pytest.skip(f"needs {G} CUDA devices")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_nccl_worker, args=(G, port, name, args, out), nprocs=G, join=True)
        return [out[r] for r in range(G)]


def _run(mode, G, name, *args):
    if mode == "threads":
        prev = torch.are_deterministic_algorithms_enabled()
        torch.use_deterministic_algorithms(True)
        try:
            res = _threads(G, CASES[name], *args)
        finally:
            torch.use_deterministic_algorithms(prev)
    else:
        res = _nccl(G, name, *args)
    bad = [f for r in res for f in r]
    assert not bad, bad


# -- cases: each returns the list of its mismatches on this rank -------------------------------------------------------
_STATES, _STATE_LOCK = {}, threading.Lock()


def _once(key, make):
    """Weights are made once per process: their initialisers draw from torch's global RNG, which the rank threads
    share -- made concurrently, each rank could get different weights."""
    with _STATE_LOCK:
        if key not in _STATES:
            _STATES[key] = make()
        return _STATES[key]


def _state(M, scale, seed=2):
    return _once(("sr", M, scale, seed), lambda: so.init_state_dict(num_maps=M, seed=seed, gain=2.3, upscale=scale))


def _vsr_state(T):
    def make():
        torch.manual_seed(0)
        return VSR(window=T).state_dict()
    return _once(("vsr", T), make)


def _stack(M, h, w, seed):
    return torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(seed)) * 255


def _nan_fill(sr):
    for ent in sr._plans.values():
        for k in ("send", "recv", "u8_band", "u8_all"):
            if k in ent:
                ent[k].view(torch.uint8).fill_(0xFF)          # NaN in every fp32 word


def case_sr(mg, dev, M, scale, h, w, cap_below, changed):
    bad = []
    sd = _state(M, scale)
    one = SRProjectionModule(num_maps=M, upscale_factor=scale)
    one.load_state_dict(sd)
    cap = None
    if cap_below:           # a cap one byte under the smallest range's unchunked workspace: every range is swept in
        from video_super_resolution_b200 import _lib       # chunks
        import ctypes
        L = _lib.lib()
        sizes = []
        for m0, m1 in map_ranges(M, mg.size):
            plan = ctypes.c_void_p()
            cfg = _lib.SrfbnConfig(M, h, w, 3, 6, 32, scale)
            _lib.check(L.vsr_srfbn_plan_create(ctypes.byref(cfg), ctypes.byref(plan)))
            _lib.check(L.vsr_srfbn_plan_set_map_range(plan, m0, m1))
            sizes.append(L.vsr_srfbn_workspace_bytes(plan))
            L.vsr_srfbn_plan_destroy(plan)
        cap = min(sizes) - 1
    sr = SRProjectionModule(num_maps=M, upscale_factor=scale, workspace_cap_bytes=cap, map_group=mg)
    sr.load_state_dict(sd)
    H, W = scale * h, scale * w
    x = _stack(M, h, w, 7).to(dev)
    want_u8 = torch.zeros((H, W, 3), dtype=torch.uint8, device=dev)
    want = one(x, out_u8=want_u8)
    u8 = torch.zeros((H, W, 3), dtype=torch.uint8, device=dev)
    sr(x, out_u8=u8)                                           # plans and exchange buffers exist from here on
    if cap_below:
        ent = [e for e in sr._plans.values() if "send" in e][0]
        m0, m1 = map_ranges(M, mg.size)[mg.rank]
        if m1 - m0 > 1 and not ent["chunk_maps"] < m1 - m0:
            bad.append(f"rank {mg.rank}: range of {m1 - m0} maps not chunked (chunk {ent['chunk_maps']})")
    _nan_fill(sr)
    u8.fill_(0x55)
    y = sr(x, out_u8=u8)
    if not torch.equal(y, want):
        bad.append(f"rank {mg.rank}: fp32 frame differs")
    if not torch.equal(u8, want_u8) or int(u8.max()) == 0:
        bad.append(f"rank {mg.rank}: u8 frame differs")
    _, _, hb = sr.band_geometry(h)
    r = mg.rank
    _nan_fill(sr)
    band = sr(x, gather=False)
    if not torch.equal(band, want[:, :, hb[r]:hb[r + 1]]):
        bad.append(f"rank {r}: fp32 band differs")
    u8b = torch.zeros_like(u8)
    sr(x, out_u8=u8b, want_f32=False, gather=False)            # only this rank's rows are written
    if not torch.equal(u8b[hb[r]:hb[r + 1]], want_u8[hb[r]:hb[r + 1]]) or \
            int(u8b[:hb[r]].count_nonzero()) + int(u8b[hb[r + 1]:].count_nonzero()) != 0:
        bad.append(f"rank {r}: u8 band")
    u8c = torch.zeros_like(u8)
    band = sr(x, out_u8=u8c, gather="u8")
    if not torch.equal(u8c, want_u8) or not torch.equal(band, want[:, :, hb[r]:hb[r + 1]]):
        bad.append(f"rank {r}: gather='u8'")
    if changed:
        x2 = x.clone()
        x2[changed:] = _stack(M - changed, h, w, 9).to(dev)
        want2_u8 = torch.zeros_like(want_u8)
        want2 = one(x2, out_u8=want2_u8, changed_from=changed)
        if not torch.equal(want2, one(x2)):
            bad.append("one-GPU refresh is not a full forward")
        sr(x)
        _nan_fill(sr)
        u82 = torch.zeros_like(u8)
        y2 = sr(x2, out_u8=u82, changed_from=changed)
        if not torch.equal(y2, want2) or not torch.equal(u82, want2_u8):
            bad.append(f"rank {r}: changed_from={changed} differs")
    return bad


def _inputs(T, h, w, seed, dev):
    la, lb = syn.logits(h, w, seed=seed + 3)
    return [t.to(dev) for t in (syn.frames(T, h, w, seed=seed), syn.smooth_flow(T - 1, h, w, 5.0, seed=seed + 1),
                                syn.inv_depth(T - 1, h, w, seed=seed + 2), la, lb)]


def case_pipe(mg, dev, T, scale, h, w, reuse, steps):
    """Deterministic projection (the caller sets the flag): each step bit-identical to the one-GPU step; step k > 0
    takes step k-1's output as its estimate (banded on the group, the full fp32 frame on one GPU)."""
    bad = []
    M = 3 * T - 1
    one = SRProjectionModule(num_maps=M, upscale_factor=scale)
    one.load_state_dict(_state(M, scale))
    sr = SRProjectionModule(num_maps=M, upscale_factor=scale, map_group=mg)
    sr.load_state_dict(_state(M, scale))
    p1 = WarpFusePipeline(T, h, w, one, scale, device=dev, reuse=reuse)
    pg = WarpFusePipeline(T, h, w, sr, scale, device=dev, reuse=reuse, map_group=mg)
    prev, band = None, None
    for k in range(steps):
        a = _inputs(T, h, w, 20 + k, dev)
        want_u8 = torch.zeros((scale * h, scale * w, 3), dtype=torch.uint8, device=dev)
        want = p1.step(*a, estimate_hr=None if prev is None else prev[0], out_u8=want_u8)
        u8 = torch.zeros_like(want_u8)
        y = pg.step(*a, estimate_hr=None if prev is None else prev[0], out_u8=u8)
        if not torch.equal(y, want) or not torch.equal(u8, want_u8):
            bad.append(f"rank {mg.rank} step {k} reuse={reuse}: full-frame step differs")
        u8b = torch.zeros_like(want_u8)
        band = pg.step(*a, estimate_hr_band=band, out_u8=u8b, gather="u8")
        if not torch.equal(u8b, want_u8):
            bad.append(f"rank {mg.rank} step {k} reuse={reuse}: banded-estimate step differs")
        prev = want
    return bad


def case_pipe_atomic(mg, dev, T, scale, h, w):
    """Default (atomic) projection: rank 0's stack is the one every rank convolves.  Returns this rank's frame and, on
    rank 0, the broadcast stack (its estimate slot restored to the fallback frame) and mask."""
    M = 3 * T - 1
    sr = SRProjectionModule(num_maps=M, upscale_factor=scale, map_group=mg)
    sr.load_state_dict(_state(M, scale))
    pg = WarpFusePipeline(T, h, w, sr, scale, device=dev, map_group=mg)
    a = _inputs(T, h, w, 31, dev)
    y = pg.step(*a)
    stack = pg.stack.clone()
    stack[M - 1] = a[0][0].permute(2, 0, 1)            # the slot before pass 1: LR frame 0 (no estimate given)
    return [("out", y.cpu(), stack.cpu() if mg.rank == 0 else None, pg._mask_w[0].cpu() if mg.rank == 0 else None)]


def _video(n, h, w, dev):
    frames = syn.frames(n, h, w, seed=1).to(dev)
    flows = syn.smooth_flow(n - 1, h, w, 2.0, seed=2).to(dev)
    inv = syn.inv_depth(n - 1, h, w, seed=3).to(dev)
    la, lb = (t.to(dev) for t in syn.logits(h, w, seed=4))
    logits = [(la + 0.1 * k, lb - 0.05 * k) for k in range(n)]
    return frames, flows, inv, logits


def case_sequence(mg, dev, n, T, h, w, split):
    frames, flows, inv, logits = _video(n, h, w, dev)
    chunks = chunk_windows(n, T, splitvideonum=split)
    one = VSR(window=T)
    one.load_state_dict(_vsr_state(T))
    want, idx = run_sequence(one, frames, flows, inv, lambda k: logits[k], chunks)
    vsr = VSR(window=T, map_group=mg)
    vsr.load_state_dict(one.state_dict())
    got, idx2 = run_sequence(vsr, frames, flows, inv, lambda k: logits[k], chunks, map_group=mg)
    if idx2 != idx or not torch.equal(got, want):
        return [f"rank {mg.rank}: run_sequence differs"]
    return []


def case_groups(pg_world, dev, n, T, h, w, split, G):
    """groups x G ranks: shard_chunks over the groups, each group map-parallel over its chunks."""
    gi, pg, ng = new_map_groups(G)
    frames, flows, inv, logits = _video(n, h, w, dev)
    chunks = shard_chunks(chunk_windows(n, T, splitvideonum=split), ng, gi)
    one = VSR(window=T)
    one.load_state_dict(_vsr_state(T))
    want, idx = run_sequence(one, frames, flows, inv, lambda k: logits[k], chunks)
    vsr = VSR(window=T, map_group=pg)
    vsr.load_state_dict(one.state_dict())
    got, idx2 = run_sequence(vsr, frames, flows, inv, lambda k: logits[k], chunks, map_group=pg)
    if idx2 != idx or not torch.equal(got, want) or not idx:
        return [f"rank {dist.get_rank()}: group {gi} run_sequence differs"]
    return []


CASES = {"sr": case_sr, "pipe": case_pipe, "sequence": case_sequence, "groups": case_groups}

MODES = ["threads", "nccl"]
SR_CASES = [  # M, scale, h, w, cap_below, changed
    (8, 4, 9, 7, False, 3),          # 9 LR rows: bands of 5 / 4 (G = 2), 3 / 3 / 3 (G = 3)
    (20, 4, 10, 6, False, 7),        # 10 rows over 3 ranks: 4 / 3 / 3; 7 / 7 / 6 maps
    (20, 4, 9, 5, True, 0),          # workspace cap: the ranges are swept in chunks
    (8, 2, 11, 6, False, 3),         # x2
    (14, 2, 8, 8, True, 0),
]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("G", [1, 2, 3])
@pytest.mark.parametrize("case", SR_CASES)
def test_sr_stack_bit_identical(mode, G, case):
    _run(mode, G, "sr", *case)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("G", [2, 3])
@pytest.mark.parametrize("reuse", [None, "frames", "unchanged"])
@pytest.mark.parametrize("T,scale,h,w", [(3, 4, 13, 20), (5, 2, 9, 16)])
def test_pipeline_step_bit_identical(mode, G, reuse, T, scale, h, w):
    _run(mode, G, "pipe", T, scale, h, w, reuse, 2)


def test_pipeline_atomic_projection_uses_rank0_stack():
    """Without the deterministic flag: every rank's frame equals every other rank's and the one-GPU two-pass run on the
    stack rank 0 broadcast."""
    T, scale, h, w = 3, 4, 13, 20
    M = 3 * T - 1
    res = _threads(3, case_pipe_atomic, T, scale, h, w)
    frames = [r[0][1] for r in res]
    assert all(torch.equal(f, frames[0]) for f in frames[1:])
    stack, mask = res[0][0][2].cuda(), res[0][0][3].cuda()
    one = SRProjectionModule(num_maps=M, upscale_factor=scale)
    one.load_state_dict(_state(M, scale))
    out1 = one(stack)
    ops.estimate_slot(out1[0], mask, stack[M - 1], scale)
    assert torch.equal(one(stack).cpu(), frames[0])


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("G", [2, 3])
def test_run_sequence_bit_identical(mode, G):
    _run(mode, G, "sequence", 14, 3, 12, 16, 2)


def test_groups_of_two_on_four_devices():
    _run("nccl", 4, "groups", 14, 3, 12, 16, 2, 2)


@pytest.mark.parametrize("mode", MODES)
def test_c2_step_two_ranks(mode):
    """C2's frame (480x270 -> 1920x1080, T = 7, M = 20) on 2 ranks: the band boundary at HR row 540, 25 MB per map
    exchanged."""
    _run(mode, 2, "pipe", 7, 4, 270, 480, None, 1)
