"""GPU: the front ops take one frame window, or W windows through a leading dimension, in one launch.  For warp_window,
compose_flow, warp_labels, vos_threshold, assemble_stack and estimate_slot: a W-window call equals W one-window calls
bit for bit, the form without a leading dimension equals the form with a leading 1, strided window views give the bits
of contiguous copies, and bad arguments raise before anything is launched.  What the ops compute is pinned against the
CPU oracle in test_pipeline_gpu and test_ops_gpu."""
import pytest
import torch

from video_super_resolution_b200 import _lib, ops, synthetic as syn

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
WINDOWS = (1, 2, 3)
SIZES = [(16, 24), (13, 19)]           # the odd size leaves a scalar tail in the vectorised kernels
T, CENTRE = 4, 2


def _once(fn):
    """fn(), which must launch exactly one kernel of the library."""
    before = _lib.launch_count()
    out = fn()
    assert _lib.launch_count() == before + 1
    return out


def _refused(exc, fn):
    before = _lib.launch_count()
    with pytest.raises(exc):
        fn()
    assert _lib.launch_count() == before


def _rand(shape, seed, scale=255.0):
    return (torch.rand(shape, generator=torch.Generator().manual_seed(seed)) * scale).to(DEV)


def _flows(nw, h, w, seed):
    """(nw,T-1,h,w,2): neighbour n of every window is the strided view x[:, n]."""
    return syn.smooth_flow(nw * (T - 1), h, w, 6.0, seed=seed).view(nw, T - 1, h, w, 2).to(DEV)


@pytest.mark.parametrize("hw", SIZES)
@pytest.mark.parametrize("nw", WINDOWS)
def test_warp_window(nw, hw):
    h, w = hw
    frames = torch.stack([syn.frames(T, h, w, seed=b) for b in range(nw)]).to(DEV)
    flows = _flows(nw, h, w, seed=10)
    warped, resid = _once(lambda: ops.warp_window(frames, flows, CENTRE))
    assert warped.shape == (nw, T - 1, h, w, 3) and resid.shape == (nw, T - 1, h, w)
    only, none = _once(lambda: ops.warp_window(frames, flows, CENTRE, want_resid=False))
    assert none is None and torch.equal(only, warped)
    for b in range(nw):
        w1, r1 = _once(lambda: ops.warp_window(frames[b], flows[b], CENTRE))
        assert torch.equal(w1, warped[b]) and torch.equal(r1, resid[b])
        w2, r2 = _once(lambda: ops.warp_window(frames[b:b + 1], flows[b:b + 1], CENTRE))
        assert w2.shape == (1,) + w1.shape and torch.equal(w2[0], w1) and torch.equal(r2[0], r1)

    _refused(ValueError, lambda: ops.warp_window(frames, flows[:, 1:], CENTRE))
    _refused(ValueError, lambda: ops.warp_window(frames, flows, T))
    _refused(ValueError, lambda: ops.warp_window(frames[None], flows[None], CENTRE))
    _refused(ValueError, lambda: ops.warp_window(frames[..., :2].contiguous(), flows, CENTRE))
    _refused(ValueError, lambda: ops.warp_window(frames.transpose(-2, -3), flows, CENTRE))
    _refused(TypeError, lambda: ops.warp_window(frames.double(), flows, CENTRE))


@pytest.mark.parametrize("hw", SIZES)
@pytest.mark.parametrize("nw", WINDOWS)
def test_compose_flow(nw, hw):
    h, w = hw
    g, f = _flows(nw, h, w, seed=20), _flows(nw, h, w, seed=30)
    out = torch.full_like(g, float("nan"))
    n = 1
    got = _once(lambda: ops.compose_flow(g[:, n], f[:, n], out=out[:, n]))
    assert got is not None and got.data_ptr() == out[:, n].data_ptr()
    gc, fc = g[:, n].contiguous(), f[:, n].contiguous()
    want = _once(lambda: ops.compose_flow(gc, fc))
    assert torch.equal(out[:, n], want)
    assert out[:, 0].isnan().all() and out[:, 2].isnan().all()                # the other neighbours are untouched
    alloc = _once(lambda: ops.compose_flow(g[:, n], f[:, n]))                 # out=None: f's window stride
    assert torch.equal(alloc, want)
    # g=None is the identity field
    assert torch.equal(_once(lambda: ops.compose_flow(None, f[:, n])), ops.compose_flow(torch.zeros_like(fc), fc))
    for b in range(nw):
        one = _once(lambda: ops.compose_flow(gc[b], fc[b]))
        assert one.shape == (h, w, 2) and torch.equal(one, want[b])
        lead = _once(lambda: ops.compose_flow(gc[b:b + 1], fc[b:b + 1]))
        assert torch.equal(lead[0], one)

    _refused(ValueError, lambda: ops.compose_flow(gc, fc[..., :1].contiguous()))
    _refused(ValueError, lambda: ops.compose_flow(gc[:, :-1].contiguous(), fc))
    _refused(ValueError, lambda: ops.compose_flow(gc, fc[None]))
    _refused(ValueError, lambda: ops.compose_flow(gc, fc.transpose(-2, -3)))          # a field that is not contiguous
    _refused(TypeError, lambda: ops.compose_flow(gc, fc.double()))
    _refused(TypeError, lambda: ops.compose_flow(gc.double(), fc))
    if nw > 1:
        _refused(ValueError, lambda: ops.compose_flow(gc, f[:, n]))                   # window strides differ
        _refused(ValueError, lambda: ops.compose_flow(None, f[:, n], out=torch.empty_like(fc)))
        odd = torch.empty(nw * (h * w * 2 + 1), device=DEV).as_strided((nw, h, w, 2), (h * w * 2 + 1, w * 2, 2, 1))
        _refused(_lib.VsrError, lambda: ops.compose_flow(None, odd, out=odd))       # an odd window stride


@pytest.mark.parametrize("hw", SIZES)
@pytest.mark.parametrize("nw", WINDOWS)
def test_warp_labels(nw, hw):
    h, w = hw
    lab = syn.labels(nw, h, w, seed=40).to(DEV)
    flows = _flows(nw, h, w, seed=50) * 2
    n = 1
    view, flat = flows[:, n], flows[:, n].contiguous()
    want = _once(lambda: ops.warp_labels(lab, flat))
    assert torch.equal(_once(lambda: ops.warp_labels(lab, view)), want)
    out = torch.full_like(lab, 7)
    assert _once(lambda: ops.warp_labels(lab, view, out=out)) is out and torch.equal(out, want)
    for b in range(nw):
        assert torch.equal(_once(lambda: ops.warp_labels(lab[b:b + 1], flat[b:b + 1])), want[b:b + 1])
        assert torch.equal(_once(lambda: ops.warp_labels(lab[b:b + 1], view[b:b + 1])), want[b:b + 1])

    _refused(ValueError, lambda: ops.warp_labels(lab, flat[:, :-1].contiguous()))
    _refused(ValueError, lambda: ops.warp_labels(lab[0], flat[0]))
    _refused(ValueError, lambda: ops.warp_labels(lab, flat.transpose(-2, -3)))
    _refused(ValueError, lambda: ops.warp_labels(lab, flat, out=torch.empty_like(lab[:, 1:])))
    _refused(TypeError, lambda: ops.warp_labels(lab.float(), flat))
    _refused(TypeError, lambda: ops.warp_labels(lab, flat.double()))
    _refused(TypeError, lambda: ops.warp_labels(lab, flat, out=torch.empty_like(lab, dtype=torch.int32)))
    if nw > 1:
        odd = torch.empty(nw * (h * w * 2 + 1), device=DEV).as_strided((nw, h, w, 2), (h * w * 2 + 1, w * 2, 2, 1))
        _refused(_lib.VsrError, lambda: ops.warp_labels(lab, odd))


@pytest.mark.parametrize("hw", SIZES)
@pytest.mark.parametrize("nw", WINDOWS)
def test_vos_threshold(nw, hw):
    h, w = hw
    pairs = [syn.logits(h, w, seed=60 + b) for b in range(nw)]
    la, lb = (torch.stack(list(x)).to(DEV) for x in zip(*pairs))
    mask = _once(lambda: ops.vos_threshold(la, lb))
    assert mask.shape == (nw, h, w) and mask.dtype == torch.uint8
    for b in range(nw):
        one = _once(lambda: ops.vos_threshold(la[b], lb[b]))
        assert one.shape == (h, w) and torch.equal(one, mask[b])
        assert torch.equal(_once(lambda: ops.vos_threshold(la[b:b + 1], lb[b:b + 1])), mask[b:b + 1])

    _refused(ValueError, lambda: ops.vos_threshold(la, lb[:, 1:].contiguous()))
    _refused(ValueError, lambda: ops.vos_threshold(la[None], lb[None]))
    _refused(ValueError, lambda: ops.vos_threshold(la, lb.transpose(-1, -2)))
    _refused(TypeError, lambda: ops.vos_threshold(la, lb.double()))


@pytest.mark.parametrize("hw", SIZES)
@pytest.mark.parametrize("nw", WINDOWS)
def test_assemble_stack(nw, hw):
    h, w = hw
    M = 3 * T - 1
    frames = _rand((nw, T, h, w, 3), 70)
    warped, proj = _rand((nw, T - 1, h, w, 3), 71), _rand((nw, T - 1, h, w, 2), 72, 16.0)
    resid, depth, est = _rand((nw, T - 1, h, w), 73), _rand((nw, T - 1, h, w), 74, 1.0), _rand((nw, 3, h, w), 75)
    for e in (None, est):
        stack = _once(lambda: ops.assemble_stack(warped, frames, proj, resid, depth, e, CENTRE))
        assert stack.shape == (nw, M, 3, h, w)
        into = torch.full_like(stack, float("nan"))
        assert _once(lambda: ops.assemble_stack(warped, frames, proj, resid, depth, e, CENTRE, out=into)) is into
        assert torch.equal(into, stack)
        for b in range(nw):
            assert torch.equal(stack[b, CENTRE], frames[b, CENTRE].permute(2, 0, 1))
            # without an estimate the slot holds LR frame 0 of the window (video_super_resolution.py:37-38)
            assert torch.equal(stack[b, M - 1], (frames[b, 0].permute(2, 0, 1) if e is None else est[b]))
            one = _once(lambda: ops.assemble_stack(warped[b], frames[b], proj[b], resid[b], depth[b],
                                                   None if e is None else e[b], CENTRE))
            assert one.shape == (M, 3, h, w) and torch.equal(one, stack[b])
            lead = _once(lambda: ops.assemble_stack(warped[b:b + 1], frames[b:b + 1], proj[b:b + 1], resid[b:b + 1],
                                                    depth[b:b + 1], None if e is None else e[b:b + 1], CENTRE))
            assert torch.equal(lead[0], one)

    args = [warped, frames, proj, resid, depth, est, CENTRE]

    def bad(i, v, **kw):
        a = list(args)
        a[i] = v
        return lambda: ops.assemble_stack(*a, **kw)
    _refused(ValueError, lambda: ops.assemble_stack(*[torch.zeros(1, device=DEV)] * 5, None, 1))
    _refused(ValueError, bad(0, warped[:, 1:].contiguous()))
    _refused(ValueError, bad(2, proj[..., :1].contiguous()))
    _refused(ValueError, bad(4, depth[None]))
    _refused(ValueError, bad(5, est[:, :2].contiguous()))
    _refused(ValueError, bad(6, T))
    _refused(ValueError, bad(1, frames.transpose(-2, -3)))
    _refused(ValueError, bad(6, CENTRE, out=torch.empty((nw, M - 1, 3, h, w), device=DEV)))
    _refused(TypeError, bad(3, resid.double()))
    _refused(TypeError, bad(6, CENTRE, out=torch.empty((nw, M, 3, h, w), device=DEV, dtype=torch.float64)))


@pytest.mark.parametrize("hw", SIZES)
@pytest.mark.parametrize("nw", WINDOWS)
def test_estimate_slot(nw, hw):
    h, w = hw
    M, s = 5, 4
    hr = _rand((nw, 3, s * h, s * w), 80)
    mask = (_rand((nw, h, w), 81, 1.0) > 0.6).to(torch.uint8)
    for m in (None, mask):
        stack = torch.full((nw, M, 3, h, w), float("nan"), device=DEV)
        assert _once(lambda: ops.estimate_slot(hr, m, stack[:, M - 1], s)).data_ptr() == stack[:, M - 1].data_ptr()
        want = _once(lambda: ops.estimate_slot(hr, m, torch.empty((nw, 3, h, w), device=DEV), s))
        assert torch.equal(stack[:, M - 1], want)
        assert stack[:, :M - 1].isnan().all()                                 # only the slot is written
        for b in range(nw):
            mb = None if m is None else m[b]
            one = _once(lambda: ops.estimate_slot(hr[b], mb, torch.empty((3, h, w), device=DEV), s))
            assert torch.equal(one, want[b])
            lead = _once(lambda: ops.estimate_slot(hr[b:b + 1], None if m is None else m[b:b + 1],
                                                   torch.empty((1, 3, h, w), device=DEV), s))
            assert torch.equal(lead[0], one)

    slot = torch.empty((nw, 3, h, w), device=DEV)
    _refused(ValueError, lambda: ops.estimate_slot(hr, mask, slot, 2))
    _refused(ValueError, lambda: ops.estimate_slot(hr, mask[:, 1:].contiguous(), slot, s))
    _refused(ValueError, lambda: ops.estimate_slot(hr[:, :2].contiguous(), None, slot[:, :2], s))
    _refused(ValueError, lambda: ops.estimate_slot(hr[None], None, slot[None], s))
    _refused(ValueError, lambda: ops.estimate_slot(hr, None, slot.transpose(-1, -2), s))
    _refused(TypeError, lambda: ops.estimate_slot(hr, mask.float(), slot, s))
    _refused(TypeError, lambda: ops.estimate_slot(hr.double(), None, slot, s))
