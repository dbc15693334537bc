"""The front (WarpFusePipeline a1-a5, a7) pinned to its CPU restatement at the benchmark's sizes: C2 (T = 7, 480x270,
W = 1, 2, 4 windows), C5 (T = 3, 720x360, W = 1, 3, 8) and C4 (T = 5, 1920x1080).

- Every front op is bit-identical to the restatement of the arithmetic it runs -- the fast mode of the warp and of the
  flow chain (oracle.or_warp_nhwc_fast / or_compose_flow_fast), the exact and nearest modes -- at a small ragged size and
  at sizes whose launches take two or more passes of their grid-stride loops (grid_for caps a launch at 148 * 8 * 4
  blocks of 256 threads = 1,212,416 threads).
- The flow projection is checked on every path its size and promise select (tile path with one or several tiles per
  CTA, general path, the gated fallback after a broken promise), with count and hole bit for bit and the fp32 sums held
  to a per-target bound derived from the arithmetic (`_proj_bounds`) instead of a flat 1e-3.
- The whole front: under torch.use_deterministic_algorithms(True) every output of project_and_warp equals the fast
  restatement bit for bit; on the default projection paths the integers match bit for bit, the sums meet the bound, and
  everything downstream of the pipeline's own projections is restated bit for bit from them."""
import contextlib
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.front_hooks import poison_workspaces, warp_carved
from video_super_resolution_b200 import _lib, ops, synthetic as syn
from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
from video_super_resolution_b200.pipeline import WarpFusePipeline

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
THREADS = max(1, min(32, os.cpu_count() or 1))
U = 2.0 ** -24                  # unit roundoff of fp32
PASS = 148 * 8 * 4 * 256        # threads of one full grid of an elementwise launch (grid_for)
SIZES = {"C2": (270, 480), "C5": (360, 720), "C4": (1080, 1920)}
REPORT = {}                     # worst error / bound ratio per projection case, printed by the last test


def _np(t):
    return t.detach().cpu().numpy()


def _bits_equal(got, want, what=""):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape, got.dtype, want.dtype)
    if got.dtype == np.float32:
        bad = got.view(np.uint32) != want.view(np.uint32)
    else:
        bad = got != want
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:4].tolist())


@contextlib.contextmanager
def _deterministic():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def _rand(shape, seed, scale=255.0):
    return (np.random.default_rng(seed).random(shape, dtype=np.float32) * np.float32(scale)).astype(np.float32)


def _flow(B, h, w, seed, mag=8.0):
    """Smooth +-mag px field plus +-0.5 px noise (fractions everywhere), a few samples beyond the borders."""
    f = syn.smooth_flow(B, h, w, mag, seed=seed).numpy()
    f = (f + (_rand(f.shape, seed + 1, 1.0) - np.float32(0.5))).astype(np.float32)
    f[:, 0, :8] = (-20.0, 3.25)
    f[:, -1, -8:] = (4000.5, -9.75)
    return np.ascontiguousarray(f)


# ---------------------------------------------------------------------------------------------------------------------
# 1. The ops, bit for bit, past one grid pass
# ---------------------------------------------------------------------------------------------------------------------
def _want_warp(src, flow, mode, ref):
    if ref is None:
        return orc.warp_nhwc(src, flow, mode, threads=THREADS), None
    return orc.warp_nhwc(src, flow, mode, threads=THREADS, ref=ref)


@pytest.mark.parametrize("C,B,h,w", [(3, 2, 37, 53), (3, 1, 1080, 1920), (8, 2, 37, 53), (8, 1, 1080, 1920),
                                     (32, 1, 37, 53), (32, 2, 1080, 1920), (5, 2, 37, 53), (5, 1, 1080, 1920)])
def test_warp_all_modes_bit_exact(C, B, h, w):
    """ops.warp: C = 3 (warp_nhwc3_kernel), 8 and 32 (vec4; with ref the generic kernel), 5 (generic), modes 0, 1, 2,
    with and without the fused residual.  At 1080p every kernel runs at least two passes of its loop."""
    src = _rand((B, h, w, C), C * 10 + B)
    ref = _rand((B, h, w, C), C * 10 + B + 1)
    flow = _flow(B, h, w, seed=C + B)
    if h * w > PASS:
        work = B * h * w * (C // 4 if C % 4 == 0 else 1)
        assert work > PASS
    s, f, r = (torch.from_numpy(x).to(DEV) for x in (src, flow, ref))
    for mode in (0, 1, 2):
        want, want_n = _want_warp(src, flow, mode, ref)
        _bits_equal(_np(ops.warp(s, f, mode)), want, (mode, "warped"))
        got, got_n = ops.warp(s, f, mode, ref=r)
        _bits_equal(_np(got), want, (mode, "warped with ref"))
        _bits_equal(_np(got_n), want_n, (mode, "resid"))


@pytest.mark.parametrize("B,h,w", [(1, 17, 19), (1, 1080, 1920)])
def test_warp_nhwc3_scalar_stores_bit_exact(B, h, w):
    """An output 4 bytes past a 16-byte boundary: warp_nhwc3_kernel stages through shared memory and stores element by
    element (vec_store = 0), over two passes at 1080p."""
    src, ref, flow = _rand((B, h, w, 3), 1), _rand((B, h, w, 3), 2), _flow(B, h, w, seed=3)
    s, f, r = (torch.from_numpy(x).to(DEV) for x in (src, flow, ref))
    for mode in (0, 1, 2):
        want, want_n = _want_warp(src, flow, mode, ref)
        got, _ = warp_carved(s, f, mode)
        _bits_equal(_np(got), want, (mode, "warped"))
        got, got_n = warp_carved(s, f, mode, r)
        _bits_equal(_np(got), want, (mode, "warped with ref"))
        _bits_equal(_np(got_n), want_n, (mode, "resid"))


def _want_window(frames, flows, centre, mode):
    """One window of ops.warp_window: neighbours in frame order with the centre left out, each compared with the
    centre frame."""
    T = frames.shape[0]
    neigh = np.ascontiguousarray(frames[[t for t in range(T) if t != centre]])
    ref = np.broadcast_to(frames[centre], neigh.shape)
    return orc.warp_nhwc(neigh, flows, mode, threads=THREADS, ref=ref)


@pytest.mark.parametrize("cfg,T,nw", [("C4", 5, 1), ("C2", 7, 1), ("C2", 7, 4), ("C5", 3, 3), ("ragged", 4, 2)])
def test_warp_window_all_modes_bit_exact(cfg, T, nw):
    """ops.warp_window at the benchmark's windows; C4's (T = 5, 1080p: 8.3 M pixels) takes seven passes, the lookahead
    flow load and both staging buffers included.  The ragged case: two windows whose outputs are not whole 16-byte
    vectors, so every window takes the scalar stores."""
    h, w = SIZES.get(cfg, (37, 53))
    c = T // 2
    frames = _rand((nw, T, h, w, 3), T * 100 + nw)
    flows = _flow(nw * (T - 1), h, w, seed=T + nw).reshape(nw, T - 1, h, w, 2)
    fr, fl = torch.from_numpy(frames).to(DEV), torch.from_numpy(flows).to(DEV)
    for mode in (0, 1, 2):
        warped, resid = ops.warp_window(fr, fl, c, mode)
        warped, resid = _np(warped), _np(resid)
        for b in range(nw):
            want, want_n = _want_window(frames[b], flows[b], c, mode)
            _bits_equal(warped[b], want, (mode, b, "warped"))
            _bits_equal(resid[b], want_n, (mode, b, "resid"))


def test_compose_flow_bit_exact_at_1080p():
    """ops.compose_flow (two passes at 1080p) against or_compose_flow_fast: one field, the identity g = None, and W = 3
    windows through the strided views x[:, n] of (3, 4, 1080, 1920, 2) arrays."""
    h, w = SIZES["C4"]
    g1, f1 = _flow(1, h, w, seed=1)[0], _flow(1, h, w, seed=2)[0]
    G, F = (torch.from_numpy(x).to(DEV) for x in (g1, f1))
    _bits_equal(_np(ops.compose_flow(G, F)), orc.compose_flow(g1, f1, fast=True, threads=THREADS), "one")
    _bits_equal(_np(ops.compose_flow(None, F)), orc.compose_flow(None, f1, fast=True, threads=THREADS), "identity")
    gw = _flow(12, h, w, seed=3).reshape(3, 4, h, w, 2)
    fw = _flow(12, h, w, seed=4).reshape(3, 4, h, w, 2)
    GW, FW = torch.from_numpy(gw).to(DEV), torch.from_numpy(fw).to(DEV)
    out = torch.full_like(GW, float("nan"))
    for n in range(4):                                            # odd n: the identity link
        ops.compose_flow(GW[:, n] if n % 2 == 0 else None, FW[:, n], out=out[:, n])
    got = _np(out)
    for b in range(3):
        for n in range(4):
            want = orc.compose_flow(gw[b, n] if n % 2 == 0 else None, fw[b, n], fast=True, threads=THREADS)
            _bits_equal(got[b, n], want, (b, n))


def test_warp_labels_bit_exact_past_one_pass():
    """B = 5 at 1080p (10.4 M pixels): the 8-pixel loop takes two passes; with the flow 8 bytes off a 16-byte boundary
    the scalar loop runs every pixel, in nine passes."""
    B, (h, w) = 5, SIZES["C4"]
    lab = syn.labels(B, h, w, seed=1).numpy()
    flow = _flow(B, h, w, seed=5)
    flow[:, 5, 5:40] = 0.5                                         # ties of floor(v + 0.5)
    want = orc.warp_labels(lab, flow)
    L = torch.from_numpy(lab).to(DEV)
    _bits_equal(_np(ops.warp_labels(L, torch.from_numpy(flow).to(DEV))), want, "aligned")
    buf = torch.empty(flow.size + 2, dtype=torch.float32, device=DEV)
    off = buf[2:].view(B, h, w, 2)
    off.copy_(torch.from_numpy(flow))
    assert off.data_ptr() % 16 == 8
    _bits_equal(_np(ops.warp_labels(L, off)), want, "flow 8 bytes off")


def test_resample2d_bit_exact_at_1080p():
    h, w = SIZES["C4"]
    img = _rand((1, 3, h, w), 7)
    flow = np.ascontiguousarray(_flow(1, h, w, seed=8).transpose(0, 3, 1, 2))
    I, F = torch.from_numpy(img).to(DEV), torch.from_numpy(flow).to(DEV)
    for bilinear in (True, False):
        _bits_equal(_np(ops.resample2d(I, F, 1, bilinear)), orc.resample2d_nchw(img, flow, 1, bilinear, threads=THREADS),
                    bilinear)


@pytest.mark.parametrize("cfg,nw,scale", [("C2", 1, 4), ("C5", 3, 4), ("C4", 1, 2)])
def test_estimate_slot_with_mask_bit_exact(cfg, nw, scale):
    h, w = SIZES[cfg]
    M = 8
    hr = _rand((nw, 3, scale * h, scale * w), 11)
    mask = (np.random.default_rng(12).random((nw, h, w)) > 0.6).astype(np.uint8)
    stack = torch.full((nw, M, 3, h, w), float("nan"), device=DEV)
    ops.estimate_slot(torch.from_numpy(hr).to(DEV), torch.from_numpy(mask).to(DEV), stack[:, M - 1], scale)
    got = _np(stack)
    for b in range(nw):
        _bits_equal(got[b, M - 1], orc.estimate_slot(hr[b], mask[b], scale), b)
    assert np.isnan(got[:, :M - 1]).all()                          # nothing else of the stack written


# ---------------------------------------------------------------------------------------------------------------------
# 2. The projection on every path, held to a per-target bound
# ---------------------------------------------------------------------------------------------------------------------
def _nearest_bound(bound, filled, axis, reverse):
    """Per pixel: bound of the nearest filled pixel before it along axis (after it with reverse), 0 where none."""
    b = np.flip(bound, axis) if reverse else bound
    f = np.flip(filled, axis) if reverse else filled
    n = b.shape[axis]
    shape = [1] * b.ndim
    shape[axis] = n
    idx = np.where(f, np.arange(n).reshape(shape), -1)
    last = np.maximum.accumulate(idx, axis=axis)
    prev = np.concatenate([np.full_like(np.take(last, [0], axis), -1), np.take(last, range(n - 1), axis)], axis)
    val = np.where(prev >= 0, np.take_along_axis(b, np.maximum(prev, 0), axis), 0.0)
    return np.flip(val, axis) if reverse else val


def _proj_bounds(flow, count, hole):
    """Per-target bounds of |proj_gpu - proj_oracle| and |wsum_gpu - wsum_oracle| / wsum_oracle, per image.

    A target with n = count hits sums n fp32 contributions c_i = round(-f_i * D_i) (and D_i) in some order: the cells'
    shared-memory or red.global additions and the 2x2 box sum together are one summation tree of n terms, so each sum
    is within (n - 1) u sum|c_i| of the exact sum (u = 2^-24), and sum|c_i| <= F sum D_i with F = max|f|.  proj = Sx / Sw
    then differs from the exact quotient by (n - 1) u F through Sx and (n - 1) u F through Sw (D_i > 0), the GPU's
    rcp.approx (1 ulp = 2u) and product (u) add 3 u F, and the oracle's own roundings -- Sx and Sw from fp64 to fp32 and
    its division -- another 3 u F:  |err| <= (2n + 4) u F, so c = 4.  wsum: (n - 1) u from the GPU's sum and u from the
    oracle's rounding of its fp64 sum, so (n + 1) u relative.  A hole takes the mean of its nearest filled neighbours
    left, right, up and down in the same order on both sides: its error is at most the largest of their bounds plus the
    roundings of three additions of values <= 4F and one division, 13 u F."""
    F = np.abs(flow.reshape(flow.shape[0], -1)).max(axis=1).reshape(-1, 1, 1).astype(np.float64)
    n = count.astype(np.float64)
    bp = (2 * n + 4) * U * F
    filled = hole == 0
    bp = np.where(filled, bp, 0.0)
    near = np.maximum.reduce([_nearest_bound(bp, filled, ax, rev) for ax in (1, 2) for rev in (False, True)])
    bp = np.where(filled, bp, near + 13 * U * F)
    return bp, (n + 1) * U


def _check_sums(case, proj, wsum, want, flow, weighted):
    """proj / wsum against the oracle's within the per-target bounds; returns the worst error / bound ratio."""
    o_proj, o_wsum, o_count, o_hole = want
    bp, bw = _proj_bounds(flow, o_count, o_hole)
    ep = np.abs(proj.astype(np.float64) - o_proj).max(axis=-1)
    ew = np.abs(wsum.astype(np.float64) - o_wsum)
    bw = bw * np.abs(o_wsum)
    assert np.isfinite(proj).all() and (ep <= bp).all(), (case, "proj", np.argwhere(ep > bp)[:4].tolist(),
                                                          float((ep / np.maximum(bp, 1e-30)).max()))
    if not weighted:
        _bits_equal(wsum, o_count.astype(np.float32), (case, "unweighted wsum is the count"))
    assert (ew <= bw).all(), (case, "wsum", np.argwhere(ew > bw)[:4].tolist())
    ratio = max(float((ep / np.maximum(bp, 1e-30)).max()), float((ew / np.maximum(bw, 1e-30)).max()))
    REPORT[case] = max(REPORT.get(case, 0.0), ratio)
    return ratio


def _n_tiles(B, h, w):
    return -(-w // 128) * -(-h // 80) * B


def _path(B, h, w, max_disp):
    """The path vsr_flow_projection_forward_bounded selects, and the library launches it takes."""
    if max_disp is None:
        return "general", 3 * B
    n = _n_tiles(B, h, w)
    if 148 < n < 148 * 7 // 4:
        return "general", 3 * B
    return ("tile, several tiles per CTA" if n > 148 else "tile, one tile per CTA"), 3


def _project(flow, inv, max_disp):
    """ops.project_flow from a poisoned workspace (the cached one of the right size exists after the first call)."""
    F = torch.from_numpy(flow).to(DEV)
    D = torch.from_numpy(inv).to(DEV) if inv is not None else None
    ops.project_flow(F, D, max_disp)                     # sizes the cached workspace
    poison_workspaces()
    torch.cuda.synchronize()
    _lib.launch_count_reset()
    out = ops.project_flow(F, D, max_disp)
    torch.cuda.synchronize()
    return [_np(t) for t in out], _lib.launch_count()


PROJ_CASES = [("C2", 1), ("C2", 2), ("C2", 4), ("C5", 1), ("C5", 3), ("C5", 8), ("C4", 1)]
PATHS_SEEN = set()


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("cfg,nw", PROJ_CASES)
def test_projection_every_path_within_the_arithmetic_bound(cfg, nw, weighted):
    """ops.project_flow at the projection batches of the benchmark's steps (B = W (T - 1) images): max_disp None (the
    general path) and 8 (the tile path, or the general path between 148 and 259 tiles), and a field that breaks the
    promise of 8 px (the tile path flags it and the gated cooperative fallback redoes the batch).  The path is asserted
    from the launch count, so a change of the path rule cannot silently drop a case."""
    T = {"C2": 7, "C5": 3, "C4": 5}[cfg]
    h, w = SIZES[cfg]
    B = nw * (T - 1)
    flow = np.ascontiguousarray(syn.smooth_flow(B, h, w, 8.0, seed=B + h).numpy())
    inv = syn.inv_depth(B, h, w, seed=B + w).numpy() if weighted else None
    want = orc.flow_projection(flow, inv, threads=THREADS)
    for md in (None, 8.0):
        path, launches = _path(B, h, w, md)
        (proj, wsum, count, hole), n = _project(flow, inv, md)
        assert n == launches, (cfg, nw, md, path, n)
        PATHS_SEEN.add(path)
        _bits_equal(count, want[2], (cfg, nw, md, "count"))
        _bits_equal(hole, want[3], (cfg, nw, md, "hole"))
        _check_sums(f"{cfg} W={nw} {'weighted' if weighted else 'plain'} {path}", proj, wsum, want, flow, weighted)
    # the broken promise: a few sources move 12 px
    broken = flow.copy()
    broken[:, h // 2, ::97, 0] = 12.0
    want_b = orc.flow_projection(broken, inv, threads=THREADS)
    path, launches = _path(B, h, w, 8.0)
    (proj, wsum, count, hole), n = _project(broken, inv, 8.0)
    assert n == launches
    _bits_equal(count, want_b[2], (cfg, nw, "broken", "count"))
    _bits_equal(hole, want_b[3], (cfg, nw, "broken", "hole"))
    name = "fallback after a broken promise" if path.startswith("tile") else path
    PATHS_SEEN.add(name)
    _check_sums(f"{cfg} W={nw} {'weighted' if weighted else 'plain'} {name}", proj, wsum, want_b, broken, weighted)


@pytest.mark.parametrize("weighted", [False, True])
def test_tile_path_cell_of_a_target_just_below_a_power_of_two(weighted):
    """Sources that land one ulp below x2 or y2 = 16, 32, 64 in the first tile column / row, where the tile's first cell
    is -1.  The tile path once took the cell as int(x2 - (-1)) in fp32, and 31.999998f + 1 rounds to 33.0f: the source
    went one cell to the right, and four targets' counts differed from the oracle's (found at C2 size, one source in
    six 480x270 smooth fields)."""
    B, h, w = 2, 90, 140
    flow = np.ascontiguousarray(syn.smooth_flow(B, h, w, 3.0, seed=9).numpy())
    k = 0
    for edge in (16, 32, 64):
        below = np.nextafter(np.float32(edge), np.float32(0))
        for b in range(B):
            y, x = 5 + 7 * k, edge - 3 + (k % 3)                  # x2 just below the edge, y2 anywhere
            flow[b, y, x, 0] = below - np.float32(x)
            assert np.float32(x) + flow[b, y, x, 0] == below
            y, x = edge - 2 + (k % 2), 70 + 5 * k                 # y2 just below the edge
            flow[b, y, x, 1] = below - np.float32(y)
            assert np.float32(y) + flow[b, y, x, 1] == below
            k += 1
    inv = syn.inv_depth(B, h, w, seed=10).numpy() if weighted else None
    want = orc.flow_projection(flow, inv, threads=THREADS)
    (proj, wsum, count, hole), n = _project(flow, inv, 8.0)
    assert n == 3                                                # the tile path
    _bits_equal(count, want[2], "count")
    _bits_equal(hole, want[3], "hole")
    _check_sums(f"cells below a power of two {'weighted' if weighted else 'plain'}", proj, wsum, want, flow, weighted)


def test_tight_bound_sees_one_source_off_by_a_thousandth_of_a_pixel():
    """Nudge one source of the oracle's input by 1e-3 px (without moving it to another cell): the per-target bound
    rejects the un-nudged GPU result against that oracle, while the flat 1e-3 bound accepts it."""
    B, (h, w) = 2, SIZES["C5"]
    flow = np.ascontiguousarray(syn.smooth_flow(B, h, w, 8.0, seed=4).numpy())
    inv = syn.inv_depth(B, h, w, seed=5).numpy()
    (proj, wsum, count, hole), _ = _project(flow, inv, 8.0)
    ys, xs = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    x2 = xs + flow[1, ..., 0]
    ok = (x2 - np.floor(x2) > 0.1) & (x2 - np.floor(x2) < 0.9) & (x2 > 2) & (x2 < w - 3)
    ok &= (ys + flow[1, ..., 1] > 2) & (ys + flow[1, ..., 1] < h - 3) & (inv[1] > 0.8)
    y, x = np.argwhere(ok)[len(np.argwhere(ok)) // 2]
    nudged = flow.copy()
    nudged[1, y, x, 0] += np.float32(1e-3)
    want = orc.flow_projection(nudged, inv, threads=THREADS)
    _bits_equal(count, want[2], "count unchanged by the nudge")
    assert np.abs(proj - want[0]).max() <= 1e-3                   # the flat bound accepts it
    with pytest.raises(AssertionError):
        _check_sums("nudged", proj, wsum, want, nudged, True)     # the per-target bound does not
    REPORT.pop("nudged", None)


# ---------------------------------------------------------------------------------------------------------------------
# 3. The whole front
# ---------------------------------------------------------------------------------------------------------------------
FRONT_CASES = [("C2", 7, 1, 4), ("C2", 7, 2, 4), ("C5", 3, 3, 4), ("C4", 5, 1, 2)]
FRONT_KEYS = ("proj_flow", "count_flow", "hole_flow", "proj_depth", "wsum", "count_depth", "hole_depth", "centre_flows",
              "warped", "resid", "mask", "mask_warped")
DOWNSTREAM = ("centre_flows", "warped", "resid", "mask", "mask_warped")


def _front_inputs(T, h, w, nw, seed):
    lead = (nw,) if nw > 1 else ()
    fr = _rand(lead + (T, h, w, 3), seed)
    fl = np.ascontiguousarray(syn.smooth_flow(nw * (T - 1), h, w, 8.0, seed=seed + 1).numpy().reshape(lead + (T - 1, h, w, 2)))
    d = syn.inv_depth(nw * (T - 1), h, w, seed=seed + 2).numpy().reshape(lead + (T - 1, h, w))
    lg = [syn.logits(h, w, seed=seed + 3 + b) for b in range(nw)]
    la = np.stack([a.numpy() for a, _ in lg]).reshape(lead + (h, w))
    lb = np.stack([b.numpy() for _, b in lg]).reshape(lead + (h, w))
    est = _rand(lead + (3, h, w), seed + 9)
    return fr, fl, d, la, lb, est


def _run_front(T, h, w, nw, scale, max_disp, inputs):
    pipe = WarpFusePipeline(T, h, w, SRProjectionModule(num_maps=3 * T - 1, upscale_factor=scale), scale, device=DEV,
                            run_fusion=False, max_disp=max_disp, windows=nw)
    poison_workspaces()
    r = pipe.project_and_warp(*(torch.from_numpy(x).to(DEV) for x in inputs))
    return {k: _np(v) for k, v in r.items()}, _np(pipe.stack)


@pytest.mark.parametrize("cfg,T,nw,scale", FRONT_CASES)
def test_front_bit_identical_to_the_fast_restatement(cfg, T, nw, scale):
    """Under torch.use_deterministic_algorithms(True) the projection is the deterministic one: every output of
    project_and_warp, and the stack, must equal orc.warp_fuse_front(..., fast=True) bit for bit."""
    h, w = SIZES[cfg]
    inputs = _front_inputs(T, h, w, nw, seed=T * 10 + nw)
    with _deterministic():
        r, stack = _run_front(T, h, w, nw, scale, None, inputs)
    want_stack, want = orc.warp_fuse_front(*inputs, threads=THREADS, fast=True)
    for k in FRONT_KEYS:
        _bits_equal(r[k], want[k], k)
    _bits_equal(stack, want_stack, "stack")


@pytest.mark.parametrize("max_disp", [None, 8.0])
@pytest.mark.parametrize("cfg,T,nw,scale", FRONT_CASES)
def test_front_on_the_default_paths(cfg, T, nw, scale, max_disp):
    """The default (atomic / tile) projection: integers bit for bit, sums within the per-target bound; then, with the
    projection taken out of the comparison, the chain, warps, label warp and assembly restated from the pipeline's own
    proj_flow / proj_depth / wsum must match bit for bit."""
    h, w = SIZES[cfg]
    inputs = _front_inputs(T, h, w, nw, seed=T * 10 + nw + 5)
    fr, fl, d = inputs[:3]
    r, stack = _run_front(T, h, w, nw, scale, max_disp, inputs)
    want_stack, want = orc.warp_fuse_front(*inputs, threads=THREADS, fast=True)
    for k in ("count_flow", "hole_flow", "count_depth", "hole_depth", "mask"):
        _bits_equal(r[k], want[k], k)
    lead = (nw * (T - 1), h, w)
    for proj_k, wsum_k, weighted, count_k, hole_k in (("proj_flow", None, False, "count_flow", "hole_flow"),
                                                      ("proj_depth", "wsum", True, "count_depth", "hole_depth")):
        wsum = r[wsum_k] if wsum_k else want[count_k].astype(np.float32)
        o_wsum = want[wsum_k] if wsum_k else want[count_k].astype(np.float32)
        _check_sums(f"front {cfg} T={T} W={nw} max_disp={max_disp} {proj_k}", r[proj_k].reshape(lead + (2,)),
                    wsum.reshape(lead), (want[proj_k].reshape(lead + (2,)), o_wsum.reshape(lead),
                                         want[count_k].reshape(lead), want[hole_k].reshape(lead)),
                    fl.reshape(lead + (2,)), weighted)
    want_stack, want = orc.warp_fuse_front(*inputs, threads=THREADS, fast=True,
                                           projected=(r["proj_flow"], r["proj_depth"], r["wsum"]))
    for k in DOWNSTREAM:
        _bits_equal(r[k], want[k], k)
    _bits_equal(stack, want_stack, "stack")


def test_report_worst_ratios_and_paths():
    """Prints the worst error / bound ratio of every projection case (run with -s), and checks that the cases above
    reached every projection path."""
    for k in sorted(REPORT):
        print(f"projection bound ratio  {REPORT[k]:.4f}  {k}")
    if REPORT:
        assert PATHS_SEEN >= {"general", "tile, one tile per CTA", "tile, several tiles per CTA",
                              "fallback after a broken promise"}, PATHS_SEEN
