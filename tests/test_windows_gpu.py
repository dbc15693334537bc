"""GPU: several frame windows per step.  A W-window step (WarpFusePipeline(windows=W)) must be bit-identical, window for
window, to W one-window steps: the front stages, both conv-stack passes (also chunked under a workspace cap and with
the fuse-pass reuse), the u8 frames, a captured graph, and the lockstep video loop (run_sequence(windows=W))."""
import contextlib

import pytest
import torch

from oracle import srfbn_oracle as so
from video_super_resolution_b200 import _lib, ops, synthetic as syn
from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
from video_super_resolution_b200.network.video_super_resolution import VSR
from video_super_resolution_b200.pipeline import GraphedStep, WarpFusePipeline, run_sequence
from video_super_resolution_b200.utils.video_utils import chunk_windows

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _sr(T, scale, cap=None):
    M = 3 * T - 1
    sr = SRProjectionModule(num_maps=M, upscale_factor=scale, workspace_cap_bytes=cap)
    sr.load_state_dict(so.init_state_dict(num_maps=M, seed=2, gain=2.3, upscale=scale))
    return sr


def _window(T, h, w, seed):
    la, lb = syn.logits(h, w, seed=seed + 3)
    return [t.to(DEV) for t in (syn.frames(T, h, w, seed=seed), syn.smooth_flow(T - 1, h, w, 5.0, seed=seed + 1),
                                syn.inv_depth(T - 1, h, w, seed=seed + 2), la, lb)]


def _batch(wins):
    return [torch.stack(list(parts)).contiguous() for parts in zip(*wins)]


@contextlib.contextmanager
def _projection_path(w):
    """The shared-memory projection path (max_disp) needs an even width; an odd width takes the deterministic path, so
    that every comparison below is between run-to-run reproducible projections."""
    if w % 2 == 0:
        yield 5.0
        return
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield None
    finally:
        torch.use_deterministic_algorithms(prev)


def _singles(T, h, w, scale, wins, reuse=None, cap=None, md=5.0):
    pipe = WarpFusePipeline(T, h, w, _sr(T, scale, cap), scale, device=DEV, max_disp=md, reuse=reuse)
    inter, ys, u8s = [], [], []
    for a in wins:
        inter.append({k: v.clone() for k, v in pipe.project_and_warp(*a).items()})
        u8 = torch.zeros((scale * h, scale * w, 3), dtype=torch.uint8, device=DEV)
        ys.append(pipe.step(*a, out_u8=u8)[0].clone())
        u8s.append(u8)
    return inter, torch.stack(ys), torch.stack(u8s)


@pytest.mark.parametrize("h,w", [(24, 40), (9, 21)])
@pytest.mark.parametrize("T,scale", [(3, 4), (7, 4), (5, 2)])
@pytest.mark.parametrize("W", [1, 2, 3, 5])
def test_batched_step_equals_single_window_steps(W, T, scale, h, w):
    wins = [_window(T, h, w, seed=10 * b + T) for b in range(W)]
    with _projection_path(w) as md:
        inter, want_y, want_u8 = _singles(T, h, w, scale, wins, md=md)
        pipe = WarpFusePipeline(T, h, w, _sr(T, scale), scale, device=DEV, max_disp=md, windows=W)
        args = _batch(wins)
        r = pipe.project_and_warp(*args)
        u8 = torch.zeros((W, scale * h, scale * w, 3), dtype=torch.uint8, device=DEV)
        y = pipe.step(*args, out_u8=u8)
    assert tuple(y.shape) == (W, 3, scale * h, scale * w)
    for k in inter[0]:
        for b in range(W):
            assert torch.equal(r[k][b], inter[b][k]), (k, b)
    assert torch.equal(y, want_y)
    assert torch.equal(u8, want_u8) and int(u8.max()) > 0


@pytest.mark.parametrize("W", [2, 3])
def test_batched_step_under_a_workspace_cap(W):
    """A cap that forces chunk_maps < W*M: the W*M maps are swept in chunks, frames unchanged."""
    T, h, w, scale = 3, 24, 40, 4
    M = 3 * T - 1
    wins = [_window(T, h, w, seed=5 * b + 1) for b in range(W)]
    _, want_y, want_u8 = _singles(T, h, w, scale, wins)
    free = _sr(T, scale)
    free(torch.zeros((W, M, 3, h, w), device=DEV))
    full = free._plans[(M, h, w, 0, W)]["workspace"].numel()
    sr = _sr(T, scale, cap=full // 2)
    pipe = WarpFusePipeline(T, h, w, sr, scale, device=DEV, max_disp=5.0, windows=W)
    u8 = torch.zeros((W, scale * h, scale * w, 3), dtype=torch.uint8, device=DEV)
    y = pipe.step(*_batch(wins), out_u8=u8)
    ent = sr._plans[(M, h, w, 0, W)]
    assert ent["chunk_maps"] < W * M and (W * M) % ent["chunk_maps"] == 0
    assert ent["workspace"].numel() <= full // 2
    assert torch.equal(y, want_y) and torch.equal(u8, want_u8)


@pytest.mark.parametrize("T", [3, 5])
def test_batched_refresh_is_bit_identical(T):
    """reuse='frames' / 'unchanged' with W windows: the fuse pass refreshes maps [first_map, M) of every window; the
    frames equal the batched reuse=None step and W one-window steps."""
    W, h, w, scale = 3, 22, 36, 4
    for seed in (7, 8):
        wins = [_window(T, h, w, seed=seed + 20 * b) for b in range(W)]
        args = _batch(wins)
        _, want_y, want_u8 = _singles(T, h, w, scale, wins)
        base = WarpFusePipeline(T, h, w, _sr(T, scale), scale, device=DEV, max_disp=5.0, windows=W)
        assert torch.equal(base.step(*args), want_y)
        for mode in ("frames", "unchanged"):
            pipe = WarpFusePipeline(T, h, w, _sr(T, scale), scale, device=DEV, max_disp=5.0, reuse=mode, windows=W)
            u8 = torch.zeros((W, scale * h, scale * w, 3), dtype=torch.uint8, device=DEV)
            for _ in range(2):                     # the second step refreshes on top of the first step's maps
                y = pipe.step(*args, out_u8=u8)
                assert torch.equal(y, want_y) and torch.equal(u8, want_u8), (mode, seed)


@pytest.mark.parametrize("W", [2, 4])
@pytest.mark.parametrize("n,T,split", [(23, 3, 4), (30, 5, 4)])
def test_run_sequence_lockstep_equals_sequential(W, n, T, split):
    h, w = 16, 24
    frames = syn.frames(n, h, w, seed=1).to(DEV)
    flows = syn.smooth_flow(n - 1, h, w, 2.0, seed=2).to(DEV)
    inv = syn.inv_depth(n - 1, h, w, seed=3).to(DEV)
    la, lb = (t.to(DEV) for t in syn.logits(h, w, seed=4))
    logits = [(la + 0.1 * k, lb - 0.05 * k) for k in range(n)]
    chunks = chunk_windows(n, T, splitvideonum=split)
    assert len({len(c) for c in chunks}) > 1                   # chunks of unequal length (one may be empty)
    torch.manual_seed(0)
    vsr = VSR(window=T)
    want, idx = run_sequence(vsr, frames, flows, inv, lambda k: logits[k], chunks)
    got, idx2 = run_sequence(vsr, frames, flows, inv, lambda k: logits[k], chunks, windows=W)
    assert idx2 == idx and got.shape == want.shape
    assert torch.equal(got, want)


def test_graphed_batched_step_replays_the_eager_frames():
    T, h, w, W = 5, 24, 40, 3
    pipe = WarpFusePipeline(T, h, w, _sr(T, 4), 4, device=DEV, max_disp=5.0, windows=W)
    g = GraphedStep(pipe, want_f32=True)
    assert tuple(g.inputs["frames"].shape) == (W, T, h, w, 3) and tuple(g.frame_u8.shape) == (W, 4 * h, 4 * w, 3)
    for seed in (3, 4):
        args = _batch([_window(T, h, w, seed=seed + 9 * b) for b in range(W)])
        u8 = torch.zeros((W, 4 * h, 4 * w, 3), dtype=torch.uint8, device=DEV)
        want = pipe.step(*args, out_u8=u8).clone()
        g.load(*args)
        got = g.replay()
        assert torch.equal(got, want) and torch.equal(g.frame_u8, u8), seed


def test_argument_errors_launch_nothing():
    T, h, w, W = 3, 16, 24, 2
    L = _lib.lib()
    with pytest.raises(ValueError):
        WarpFusePipeline(T, h, w, _sr(T, 4), 4, device=DEV, windows=0)
    pipe = WarpFusePipeline(T, h, w, _sr(T, 4), 4, device=DEV, max_disp=5.0, windows=W)
    good = _batch([_window(T, h, w, seed=b) for b in range(W)])
    pipe.step(*good)                                           # plans exist: what follows must not launch
    torch.cuda.synchronize()
    bad = [
        [good[0][:1]] + good[1:],                                            # one window of frames
        [good[0], good[1][:, :1]] + good[2:],                                # T-2 flows
        good[:3] + [good[3][0], good[4]],                                    # logits without the window dimension
        [good[0].transpose(2, 3).contiguous().transpose(2, 3)] + good[1:],   # not contiguous
    ]
    _lib.launch_count_reset()
    for args in bad:
        with pytest.raises(ValueError):
            pipe.step(*args)
    with pytest.raises(ValueError):
        pipe.step(*good, estimate_hr=torch.zeros((W, 3, h, w), device=DEV))
    with pytest.raises(ValueError):
        pipe.sr(torch.zeros((2 * pipe.M + 1, 3, h, w), device=DEV))
    with pytest.raises(ValueError):
        pipe.sr(pipe.stack, out_u8=torch.zeros((4 * h, 4 * w, 3), dtype=torch.uint8, device=DEV))
    with pytest.raises(ValueError):
        ops.warp_window(good[0], good[1][:1], 1)
    with pytest.raises(ValueError):
        ops.assemble_stack(*[torch.zeros(1, device=DEV)] * 5, None, 1)
    assert _lib.launch_count() == 0
    # the setter after bind
    ent = pipe.sr._plans[(3 * T - 1, h, w, 0, W)]
    assert L.vsr_srfbn_plan_set_windows(ent["plan"], 3) == 4                 # VSR_ERR_STATE
    assert L.vsr_srfbn_plan_set_windows(ent["plan"], 0) == 1                 # VSR_ERR_INVALID_ARG
    assert _lib.launch_count() == 0


def test_profile_counts_scale_with_windows():
    """Launches per kernel class are those of one window (the maps are swept together); FLOPs and bytes scale by W."""
    T, h, w = 3, 16, 24
    M = 3 * T - 1
    prof = {}
    for W in (1, 3):
        sr = _sr(T, 4)
        x = torch.rand((W * M, 3, h, w), generator=torch.Generator().manual_seed(1)).to(DEV) * 255
        sr(x)
        sr.profile(True)
        sr(x)
        prof[W] = sr.profile_read()
        sr.profile(False)
    for k, d in prof[1].items():
        assert prof[3][k]["launches"] == d["launches"], k
        assert prof[3][k]["flops"] == pytest.approx(3 * d["flops"], rel=1e-9), k
        assert prof[3][k]["bytes"] == pytest.approx(3 * d["bytes"], rel=1e-9), k
    # the per-map images of W windows, window-major
    sr = _sr(T, 4)
    x = torch.rand((2, M, 3, h, w), generator=torch.Generator().manual_seed(2)).to(DEV) * 255
    maps = sr.premix(x)
    assert tuple(maps.shape) == (2 * M, 3, 4 * h, 4 * w)
    assert torch.equal(maps[M:], _sr(T, 4).premix(x[1].contiguous()))
