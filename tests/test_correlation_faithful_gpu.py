"""The correlation kernels of correlation.cu pinned bit for bit to their CPU restatement (oracle.or_correlation with
padded=1, oracle.or_correlation_backward_chain; the restatement itself is checked in test_correlation_restatement):

- both forward paths (the register-tiled correlation_s2_kernel and, with VSR_CORR_GENERIC set, the generic kernel) and
  the backward at FlowNetC's size (256 x 135 x 240, pad 20, max displacement 20, strides 1 / 2), with batch items and
  channel slices that run in the first, a middle and the last pass of the grid-stride loops;
- the training crop and the edges of the geometry (channel tails, ragged x-tiles, D = 1 and 21, pad below and above the
  displacement, 3x3 and 5x5 windows, strided outputs);
- Inf and NaN in the inputs and in grad_output, at the borders and inside: the same NaN mask as the restatement (the
  reference's zero padding: 0 * Inf is NaN) and the same bits elsewhere.

Every output is first filled with a sentinel, so an element the kernels do not write is seen.  NaN payloads differ
between x86 and CUDA, so NaN is compared as a mask."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from video_super_resolution_b200 import _lib

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
THREADS = max(1, min(32, os.cpu_count() or 1))
NAN = float("nan")
FLOWNETC = (20, 1, 20, 1, 2)         # pad, kernel size, max displacement, stride1, stride2 (FlowNetC.py:22)


def _geometry(H, W, pad, k, md, s1, s2):
    border = (k - 1) // 2 + md
    R = md // s2
    return (2 * R + 1) ** 2, -(-(H + 2 * pad - 2 * border) // s1), -(-(W + 2 * pad - 2 * border) // s1)


def _forward(a, b, pad, k, md, s1, s2, sentinel=NAN):
    """vsr_correlation_forward into an output filled with `sentinel`."""
    B, C, H, W = a.shape
    out = torch.full((B,) + _geometry(H, W, pad, k, md, s1, s2), sentinel, device=DEV)
    _lib.check(_lib.lib().vsr_correlation_forward(a.data_ptr(), b.data_ptr(), out.data_ptr(), B, C, H, W, pad, k, md,
                                                  s1, s2, 1, torch.cuda.current_stream().cuda_stream), "correlation")
    torch.cuda.synchronize()
    return out


def _backward(a, b, g, pad, k, md, s2, sentinel=NAN):
    B, C, H, W = a.shape
    g1, g2 = torch.full_like(a, sentinel), torch.full_like(a, sentinel)
    _lib.check(_lib.lib().vsr_correlation_backward(a.data_ptr(), b.data_ptr(), g.data_ptr(), g1.data_ptr(), g2.data_ptr(),
                                                   B, C, H, W, pad, k, md, 1, s2, 1,
                                                   torch.cuda.current_stream().cuda_stream), "correlation_backward")
    torch.cuda.synchronize()
    return g1, g2


def _same(got, want, what):
    """Bit for bit where the restatement is not NaN, and the same NaN mask."""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), (what, "NaN mask", int((gn != wn).sum()), np.argwhere(gn != wn)[:4].tolist())
    bad = got.view(np.int32) != want.view(np.int32)
    bad &= ~wn
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:4].tolist())


def _paths(monkeypatch):
    """Yield the path name with VSR_CORR_GENERIC set accordingly (the register-tiled kernel serves k 1, s1 1, s2 2)."""
    for name in ("register-tiled", "generic"):
        if name == "generic":
            monkeypatch.setenv("VSR_CORR_GENERIC", "1")
        else:
            monkeypatch.delenv("VSR_CORR_GENERIC", raising=False)
        yield name
    monkeypatch.delenv("VSR_CORR_GENERIC", raising=False)


def _inputs(shape, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(shape, generator=g, device=DEV), torch.randn(shape, generator=g, device=DEV))


def _np(t):
    return t.detach().cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------------
# FlowNetC size
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 8])
def test_flownetc_forward_bit_for_bit_both_paths(B, monkeypatch):
    """1080p/8 features.  At B = 8 the register-tiled kernel has 8*135*21*2 = 45,360 warp tasks against 148*64 blocks
    * 4 warps = 37,888 per pass, so item 7 runs in the second pass (the generic kernel: 181,440 tasks against 75,776,
    item 7 in the third)."""
    C, H, W = 256, 135, 240
    a, b = _inputs((B, C, H, W), 100 + B)
    an, bn = _np(a), _np(b)
    items = [0] if B == 1 else [0, 7]
    if B == 8:
        assert 8 * 135 * 21 * 2 > 148 * 64 * 4 and 7 * 135 * 21 * 2 >= 148 * 64 * 4
    want = {n: orc.correlation(an, bn, *FLOWNETC, padded=True, items=(n, n + 1), threads=THREADS)[0] for n in items}
    for path in _paths(monkeypatch):
        out = _forward(a, b, *FLOWNETC)
        for n in items:
            _same(_np(out[n]), want[n], (path, B, n))
        assert not torch.isnan(out).any(), path            # every item written
        del out


def test_training_crop_forward_bit_for_bit_both_paths(monkeypatch):
    """(8, 256, 48, 64): outW = 64, one partial 128-column tile of the register-tiled kernel."""
    a, b = _inputs((8, 256, 48, 64), 7)
    want = orc.correlation(_np(a), _np(b), *FLOWNETC, padded=True, threads=THREADS)
    for path in _paths(monkeypatch):
        _same(_np(_forward(a, b, *FLOWNETC)), want, path)


def test_flownetc_backward_bit_for_bit_first_middle_last_pass():
    """(2, 256, 135, 240): 16.6 M elements per gradient against 148*64 blocks * 256 threads = 2,424,832 per pass, seven
    passes.  Channel slices of item 0 in the first pass (channels 0-7) and in the middle one (228-235: pass 3), and of
    item 1 in the last (248-255: pass 6)."""
    B, C, H, W = 2, 256, 135, 240
    per_pass, HW = 148 * 64 * 256, H * W
    a, b = _inputs((B, C, H, W), 11)
    g = torch.randn((B, 441, H, W), generator=torch.Generator(device=DEV).manual_seed(12), device=DEV)
    g1, g2 = _backward(a, b, g, 20, 1, 20, 2)
    assert not torch.isnan(g1).any() and not torch.isnan(g2).any()
    an, bn, gn = _np(a), _np(b), _np(g)
    slices = [(0, 0, 8), (0, 228, 236), (1, 248, 256)]
    assert [((n * C + c0) * HW // per_pass, ((n * C + c1) * HW - 1) // per_pass) for n, c0, c1 in slices] == \
        [(0, 0), (3, 3), (6, 6)] and (B * C * HW - 1) // per_pass == 6
    for n, c0, c1 in slices:
        w1, w2 = orc.correlation_backward_chain(an, bn, gn, 20, 1, 20, 2, items=(n, n + 1), channels=(c0, c1),
                                                threads=THREADS)
        _same(_np(g1[n:n + 1, c0:c1]), w1, ("grad_input1", n, c0))
        _same(_np(g2[n:n + 1, c0:c1]), w2, ("grad_input2", n, c0))


# ---------------------------------------------------------------------------------------------------------------------
# Edges of the geometry
# ---------------------------------------------------------------------------------------------------------------------
EDGES = [
    # (B, C, H, W), pad, k, md, s1, s2
    ((2, 9, 20, 40), 20, 1, 20, 1, 2),      # C % 8 = 1: the last staging group holds one channel
    ((1, 15, 18, 44), 20, 1, 20, 1, 2),     # C % 8 = 7
    ((1, 8, 12, 129), 4, 1, 4, 1, 2),       # outW % 128 = 1: a last tile of one column
    ((1, 8, 10, 255), 4, 1, 4, 1, 2),       # outW % 128 = 127
    ((2, 5, 9, 20), 6, 1, 6, 1, 2),         # outW < 32: one partial warp
    ((1, 6, 11, 37), 1, 1, 1, 1, 2),        # D = 1 (max displacement below stride2)
    ((1, 12, 30, 60), 21, 1, 21, 1, 2),     # D = 21 with md 21 not a multiple of s2
    ((2, 10, 40, 70), 6, 1, 10, 1, 2),      # pad < md: the output shrinks
    ((1, 10, 24, 50), 14, 1, 10, 1, 2),     # pad > md: padded rows and columns of in1 inside the output
    ((1, 7, 20, 28), 5, 3, 4, 1, 1),        # 3x3 window, pad = md + krad
    ((1, 5, 16, 21), 7, 5, 3, 1, 1),        # 5x5 window, pad > md + krad
    ((1, 6, 21, 37), 4, 1, 4, 2, 2),        # s1 = 2 (generic kernel)
    ((2, 4, 23, 31), 5, 3, 3, 3, 1),        # s1 = 3 with a 3x3 window
]


@pytest.mark.parametrize("cfg", EDGES, ids=lambda c: "x".join(map(str, c[0])) + f"-p{c[1]}k{c[2]}m{c[3]}s{c[4]}{c[5]}")
def test_geometry_edges_bit_for_bit(cfg, monkeypatch):
    shape, pad, k, md, s1, s2 = cfg
    a, b = _inputs(shape, sum(shape) + pad + md)
    an, bn = _np(a), _np(b)
    want = orc.correlation(an, bn, pad, k, md, s1, s2, padded=True, threads=THREADS)
    outs = {path: _np(_forward(a, b, pad, k, md, s1, s2)) for path in _paths(monkeypatch)}
    for path, got in outs.items():
        _same(got, want, path)
    assert np.abs(want).max() > 0
    if s1 == 1:
        g = torch.randn((shape[0],) + want.shape[1:], generator=torch.Generator(device=DEV).manual_seed(3), device=DEV)
        w1, w2 = orc.correlation_backward_chain(an, bn, _np(g), pad, k, md, s2, threads=THREADS)
        g1, g2 = _backward(a, b, g, pad, k, md, s2)
        _same(_np(g1), w1, "grad_input1")
        _same(_np(g2), w2, "grad_input2")


@pytest.mark.parametrize("md, s2", [(11, 1), (22, 2)])
def test_more_than_21_displacements_rejected_with_nothing_launched(md, s2, monkeypatch):
    """D = 23 does not fit the kernels' registers: VSR_ERR_UNSUPPORTED on both paths, no launch, output untouched."""
    a, b = _inputs((1, 4, 30, 40), 5)
    for path in _paths(monkeypatch):
        out = torch.full((1, 23 * 23) + _geometry(30, 40, md, 1, md, 1, s2)[1:], NAN, device=DEV)
        torch.cuda.synchronize()
        before = _lib.launch_count()
        rc = _lib.lib().vsr_correlation_forward(a.data_ptr(), b.data_ptr(), out.data_ptr(), 1, 4, 30, 40, md, 1, md, 1,
                                                s2, 1, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert rc == 2, (path, rc)                             # VSR_ERR_UNSUPPORTED
        assert _lib.launch_count() == before, path
        assert torch.isnan(out).all(), path


# ---------------------------------------------------------------------------------------------------------------------
# Non-finite inputs
# ---------------------------------------------------------------------------------------------------------------------
def _poison(x, seed, values):
    """Non-finite values in the first and last rows and columns and inside, in a few channels of every item."""
    B, C, H, W = x.shape
    rng = np.random.default_rng(seed)
    spots = [(0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1), (0, W // 2), (H - 1, W // 3), (H // 2, 0),
             (H // 3, W - 1), (H // 2, W // 2), (H // 3 + 1, 2 * W // 3), (5, W // 4), (H - 6, 3 * W // 4)]
    for n in range(B):
        for i, (y, xx) in enumerate(spots):
            x[n, int(rng.integers(C)), y, xx] = values[i % len(values)]
    return x


NONFINITE = [
    ((2, 19, 24, 150), 20, 1, 20, 1, 2),    # FlowNetC geometry: in2's padded rows meet in1's Inf / NaN
    ((1, 10, 24, 50), 14, 1, 10, 1, 2),     # pad > md: in1's padded rows meet in2's Inf / NaN
    ((1, 9, 30, 44), 6, 1, 10, 1, 2),       # pad < md
    ((1, 6, 18, 26), 5, 3, 4, 1, 1),        # 3x3 window
]


@pytest.mark.parametrize("cfg", NONFINITE, ids=lambda c: "x".join(map(str, c[0])) + f"-p{c[1]}k{c[2]}m{c[3]}")
def test_nonfinite_inputs_follow_the_padded_rule(cfg, monkeypatch):
    shape, pad, k, md, s1, s2 = cfg
    a, b = _inputs(shape, 40 + pad)
    a = _poison(a, 1, (float("inf"), NAN, float("-inf")))
    b = _poison(b, 2, (NAN, float("-inf"), float("inf")))
    an, bn = _np(a), _np(b)
    want = orc.correlation(an, bn, pad, k, md, s1, s2, padded=True, threads=THREADS)
    skip = orc.correlation(an, bn, pad, k, md, s1, s2, padded=False, threads=THREADS)
    assert np.isnan(want).sum() > np.isnan(skip).sum()       # the case reaches padding with a non-finite value
    assert np.isfinite(want).sum() > want.size // 2
    masks = []
    for path in _paths(monkeypatch):
        for sentinel in (NAN, 7.0):                          # a NaN the kernel failed to write would hide in a NaN
            got = _np(_forward(a, b, pad, k, md, s1, s2, sentinel))
            _same(got, want, (path, sentinel))
        masks.append(np.isnan(got))
    assert np.array_equal(masks[0], masks[1])
    g = torch.randn((shape[0],) + want.shape[1:], generator=torch.Generator(device=DEV).manual_seed(9), device=DEV)
    g = _poison(g, 3, (float("inf"), NAN))
    for ga, gb, what in ((_inputs(shape, 41)[0], _inputs(shape, 42)[1], "grad_output"), (a, b, "all")):
        w1, w2 = orc.correlation_backward_chain(_np(ga), _np(gb), _np(g), pad, k, md, s2, threads=THREADS)
        for sentinel in (NAN, 7.0):
            g1, g2 = _backward(ga, gb, g, pad, k, md, s2, sentinel)
            _same(_np(g1), w1, ("grad_input1", what, sentinel))
            _same(_np(g2), w2, ("grad_input2", what, sentinel))
