"""GPU: the bound SR plan walked one layer at a time (vsr_srfbn_debug_run_layers), each layer's output checked against the
single-layer hook fed the same inputs and the state-dict weights the SRFBN graph names for that layer, against the
BF16-faithful restatement (oracle/srfbn_bf16.py) on those inputs, and for writes into any other buffer of the workspace.

The single-layer tests build their layers themselves and the whole-stack tests cannot be tight (40-odd layers carry
BF16 rounding flips), so neither sees the plan's wiring: which buffers a layer of build_layer_list reads and writes, the
weight and bias slot it uses, where vsr_srfbn_pack_weights puts each bias and slope, and how
SRProjectionModule._weights_struct maps state-dict names.  Here a wrong source, weight, bias or slope changes the bits
of the layer that uses it, and the walk names that layer.  It also runs the layers no hook builds: the dense-concat 1x1
layers over 2-6 separate sources (one tensor map each), compress_in over xfeat twice (step 0) and over the previous
step's hidden, and, at (8, 80, 90) x4 / (8, 40, 90) x2, 1x1 layers of 450 / 900 tiles on 444 CTAs.

Two deliberately wrong builds, walked once each on a B200 and not kept: compress_out with its sources lr[2] and lr[5]
swapped in build_layer_list fails at "step 0 compress_out" (over 99 % of its outputs differ from the hook's), and
vsr_srfbn_pack_weights storing uptran_slope[i + 1] for uptran i fails at "step 0 uptranBlocks.0".  Both also fail every
case of the whole-stack restatement test; the fp32-oracle test catches the first in all its cases and the second in
its x2 cases only.

The walk covers the first chunk of an unchunked one-window plan; chunked, windowed and map-range plans are pinned bit for
bit to that plan by their own tests.  Measured on one NVIDIA B200 (1000 W power limit) the file runs in 12 s, 5.2 s
of it the (8, 80, 90) x4 walk."""
import ctypes
import math
import time

import pytest
import torch
import torch.nn.functional as F

from oracle import srfbn_bf16 as sb
from tests import srfbn_hooks as hk
from tests.srfbn_hooks import (BUF_A0, BUF_ACC, BUF_C128, BUF_HB, BUF_HIDDEN, BUF_HR, BUF_HT, BUF_LR, BUF_PREMIX, BUF_U,
                               BUF_XFEAT)
from tests.test_srfbn_faithful_gpu import MAX_DIFF_FRAC, STACK_BOUNDS, _map_errors
from tests.test_srfbn_gpu import _MAX_DIFF_FRAC_FUSED
from video_super_resolution_b200 import _lib
from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
A0, C128, XFEAT, HIDDEN, U, HB, HT, ACC, PREMIX = ((b, 0) for b in (BUF_A0, BUF_C128, BUF_XFEAT, BUF_HIDDEN, BUF_U,
                                                                    BUF_HB, BUF_HT, BUF_ACC, BUF_PREMIX))


def LR(i):
    return (BUF_LR, i)


def HR(i):
    return (BUF_HR, i)


def _d(t):
    return t.to(DEV, torch.float64)


class LayerMismatch(AssertionError):
    """The first walk step whose output fails a check; `label` names the step."""

    def __init__(self, label, msg):
        super().__init__(f"{label}: {msg}")
        self.label = label


# ---- the plan as the SRFBN graph gives it --------------------------------------------------------------------------
def _plan_steps(scale, steps):
    """[(label, kernel classes, kind, args)] in launch order, derived from the graph (SRProjectionModule.py:45-80,
    :137-145: the dense-concat dataflow, `out` and conv_out after the last step only) and the plan's one fusion rule: an
    x4 feedback group over nsrc >= 4 HR maps runs as one merged up-down launch, the others as the transposed conv and
    the fused down kernel.  The fused down kernels and their finalize_lr are one step."""
    pw, pwh, dc, dn = "pointwise_lr", "pointwise_hr", "deconv8x8s4", "conv8x8s4"
    down = ["fused_downtran_conv8x8s4", "finalize_lr"]
    seq = [("conv_in", ["conv_in_gemm"], "conv_in", {}),
           ("feat_in", [pw], "pw", dict(prefix="feat_in", srcs=[C128], out=XFEAT))]
    for t in range(steps):
        seq.append((f"step {t} compress_in", [pw], "pw",
                    dict(prefix="block.compress_in", srcs=[XFEAT, XFEAT if t == 0 else HIDDEN], out=LR(0))))
        for i in range(6):
            up_in = LR(0)
            if i > 0:
                seq.append((f"step {t} uptranBlocks.{i - 1}", [pw], "pw",
                            dict(prefix=f"block.uptranBlocks.{i - 1}", srcs=[LR(j) for j in range(i + 1)], out=U)))
                up_in = U
            if scale == 2:
                seq.append((f"step {t} upBlocks.{i}", [dc], "up",
                            dict(prefix=f"block.upBlocks.{i}", src=up_in, out=HR(i))))
                down_in = HR(0)
                if i > 0:
                    seq.append((f"step {t} downtranBlocks.{i - 1}", [pwh], "pw",
                                dict(prefix=f"block.downtranBlocks.{i - 1}", srcs=[HR(j) for j in range(i + 1)],
                                     out=HT)))
                    down_in = HT
                seq.append((f"step {t} downBlocks.{i}", [dn], "down2",
                            dict(prefix=f"block.downBlocks.{i}", src=down_in, out=LR(i + 1))))
            elif i + 1 >= 4:
                seq.append((f"step {t} merged group {i}", down, "updown", dict(group=i, up_in=up_in)))
            else:
                seq.append((f"step {t} upBlocks.{i}", [dc], "up",
                            dict(prefix=f"block.upBlocks.{i}", src=up_in, out=HR(i), block=True)))
                seq.append((f"step {t} downBlocks.{i}", down, "fused", dict(group=i)))
        seq.append((f"step {t} compress_out", [pw], "pw",
                    dict(prefix="block.compress_out", srcs=[LR(j) for j in range(1, 7)], out=HIDDEN)))
    seq.append(("out", [dc], "up", dict(prefix="out", src=HIDDEN, out=HB, block=False)))
    seq.append(("conv_out", ["conv_out3x3"], "conv_out", {}))
    return seq


def test_layer_counts_of_the_graph():
    """4 + 22 steps' worth of launches per feedback step at x4, 4 + 24 at x2 (build_layer_list at the parent commit)."""
    for scale, per in ((4, 22), (2, 24)):
        for steps in (1, 2, 3):
            assert sum(len(c) for _, c, _, _ in _plan_steps(scale, steps)) == 4 + per * steps


# ---- one plan and its workspace ------------------------------------------------------------------------------------
class _Plan:
    """SRProjectionModule bound for the maps x, its workspace buffers, the kernel classes of its layer list from a
    profiled forward, and the per-map images of a whole forward."""

    def __init__(self, sd, M, h, w, steps, scale):
        self.M, self.h, self.w, self.steps, self.s = M, h, w, steps, scale
        self.mod = SRProjectionModule(num_steps=steps, num_maps=M, upscale_factor=scale)
        self.mod.load_state_dict(sd)
        self.x = (torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(5)) * 255).to(DEV)
        self.ent = self.mod._plan_for(M, h, w, torch.device(DEV))
        assert self.ent["chunk_maps"] == M
        self.views, self.ranges = self._buffers()
        self.classes = self._profiled_classes()
        self.premix = self.mod.premix(self.x).clone()
        self.frame = self.mod(self.x).clone()

    def _buffers(self):
        M, h, w, s = self.M, self.h, self.w, self.s
        bf, lr = torch.bfloat16, (M, h, w, 32)
        hr = (M, 2 * h, 2 * w, 32) if s == 2 else (M, 8, h + 1, w + 1, 64)
        shapes = {A0: ((M * h * w, 32), bf), C128: ((M, h, w, 128), bf), XFEAT: (lr, bf), HIDDEN: (lr, bf),
                  U: (lr, bf), HB: ((M, s * h, s * w, 32), bf), PREMIX: ((M, 3, s * h, s * w), torch.float32)}
        shapes.update({LR(i): (lr, bf) for i in range(7)})
        shapes.update({HR(i): (hr, bf) for i in range(6 if s == 2 else 5)})   # x4 hr[5] stays on chip
        shapes.update({HT: (hr, bf)} if s == 2 else {ACC: ((M * h * w * 128,), torch.float32)})
        views, ranges = {}, {}
        for (b, i), (shape, dt) in shapes.items():
            v = hk.plan_buffer(self.ent, b, i, shape, dt)
            views[(b, i)] = v
            ranges[(b, i)] = (v.data_ptr() - self.ent["workspace"].data_ptr(), v.numel() * v.element_size())
        return views, ranges

    def _profiled_classes(self):
        L = _lib.lib()
        self.mod.profile(True)
        self.mod(self.x)
        cap = 4096
        ms, kc = (ctypes.c_float * cap)(), (ctypes.c_int32 * cap)()
        n = L.vsr_srfbn_profile_launches(self.ent["plan"], ms, kc, cap)
        self.mod.profile(False)
        assert 2 < n <= cap, n
        names = [L.vsr_srfbn_kernel_class_name(kc[i]).decode() for i in range(n)]
        assert names[0] == "im2col" and names[-1] == "fc_fuse", names
        return names[1:-1]


def _faithful(got, want, absdot, what, max_frac, **kw):
    """hk.faithful_bf16 with the single-layer tests' per-element bound, and their fraction bound rounded up to a whole
    number of elements: ceil(max_frac * n) of n outputs may differ.  The single-layer tests' outputs are large enough
    for that to be max_frac; layers of the walk's 1 x 1, 13 x 1 and 1 x 17 cases have from 64 outputs, where max_frac
    allows a fraction of one element and two flips in one layer are a matter of chance, not of wiring."""
    n = got.numel()
    return hk.faithful_bf16(got, want, absdot, what, max_frac=math.ceil(max_frac * n) / n, **kw)


def _ring_zero(blk, what):
    """The zero ring of an HR block-layout map: every element outside the image is 0."""
    B, _, hb, wb, _ = blk.shape
    ring = hk.to_block(torch.ones((B, 4 * (hb - 1), 4 * (wb - 1), 32), device=blk.device)) == 0
    assert bool((blk.float()[ring] == 0).all()), f"{what}: the zero ring of the HR block layout is not zero"


# ---- one step's checks ---------------------------------------------------------------------------------------------
class _Checks:
    """Hook identity and restatement agreement of one step, with the expected side's state dict and restatement."""

    def __init__(self, plan, sd, R):
        self.p, self.sd, self.R = plan, sd, R

    def w(self, prefix):
        return self.sd[prefix + ".0.weight"]

    def b(self, prefix):
        return self.sd[prefix + ".0.bias"]

    def slope(self, prefix):
        return float(self.sd[prefix + ".1.weight"].reshape(-1)[0])

    def rw(self, prefix):
        return self.R.weight(self.sd, prefix, DEV)

    def conv_in(self, inp, label):
        sd, R, x = self.sd, self.R, self.p.x
        got = self.p.views[C128]
        hk.bits_equal(got, hk.conv_in(x, self.w("conv_in"), self.b("conv_in"), self.slope("conv_in"),
                                      sd["sub_mean.bias"]), f"{label} vs vsr_test_conv_in")
        want = R.conv_in(_d(x), sd).permute(0, 2, 3, 1)
        xs = R.rb(_d(x) + _d(sd["sub_mean.bias"]).view(1, 3, 1, 1))
        w, b = self.rw("conv_in"), _d(self.b("conv_in"))
        pre = F.conv2d(xs, w, b, padding=1).permute(0, 2, 3, 1)
        absdot = F.conv2d(xs.abs(), w.abs(), b.abs(), padding=1).permute(0, 2, 3, 1)
        _faithful(got, want, absdot, label, MAX_DIFF_FRAC, ulps=hk.ulps(want, pre=pre))

    def pw(self, inp, label, prefix, srcs, out):
        xin = torch.cat([inp[k] for k in srcs], dim=-1)
        xin = xin.reshape(-1, xin.shape[-1])                 # (rows, K): the channel concatenation of the sources
        got = self.p.views[out].reshape(-1, 32)
        hk.bits_equal(got, hk.pointwise(xin, self.w(prefix).view(32, -1), self.b(prefix), self.slope(prefix)),
                      f"{label} vs vsr_test_pointwise", dims="row,c")
        xd, wd, bd = _d(xin), self.rw(prefix).view(32, -1), _d(self.b(prefix))
        pre = xd @ wd.t() + bd
        want = self.R.act_packed(pre, self.sd, prefix)
        _faithful(got, want, xd.abs() @ wd.abs().t() + bd.abs(), label, MAX_DIFF_FRAC, ulps=hk.ulps(want, pre=pre))

    def up(self, inp, label, prefix, src, out, block=False):
        """A transposed conv on its own launch: x4 into the HR block layout (block) or plain NHWC (`out`), or x2."""
        s, xin, got = self.p.s, inp[src], self.p.views[out]
        if s == 2:
            hook = hk.x2_layer(xin, self.w(prefix), self.b(prefix), self.slope(prefix), up=True)
        else:
            hook = hk.deconv(xin, self.w(prefix), self.b(prefix), self.slope(prefix), block_layout=block)
        hk.bits_equal(got, hook, f"{label} vs the transposed-conv hook", dims="b,pair,Yb,Xb,el" if block else "b,y,x,c")
        if block:
            _ring_zero(got, label)
            got = hk.from_block(got)
        self._up_faithful(_d(xin), got, label, prefix)

    def _up_faithful(self, xd, got, label, prefix):
        _, st, pd = sb.GEOMETRY[self.p.s]
        xc, wd, bd = xd.permute(0, 3, 1, 2), self.rw(prefix), _d(self.b(prefix))
        want = self.R.up(xc, self.sd, prefix, self.p.s).permute(0, 2, 3, 1)
        pre = F.conv_transpose2d(xc, wd, bd, stride=st, padding=pd).permute(0, 2, 3, 1)
        absdot = F.conv_transpose2d(xc.abs(), wd.abs(), bd.abs(), stride=st, padding=pd).permute(0, 2, 3, 1)
        _faithful(got, want, absdot, label, MAX_DIFF_FRAC, ulps=hk.ulps(want, pre=pre))

    def down2(self, inp, label, prefix, src, out):
        xin, got = inp[src], self.p.views[out]
        hook = hk.x2_layer(xin, self.w(prefix), self.b(prefix), self.slope(prefix), up=False)
        hk.bits_equal(got, hook, f"{label} vs vsr_test_x2_layer")
        xc, wd, bd = _d(xin).permute(0, 3, 1, 2), self.rw(prefix), _d(self.b(prefix))
        want = self.R.down(xc, self.sd, prefix, 2).permute(0, 2, 3, 1)
        pre = F.conv2d(xc, wd, bd, stride=2, padding=2).permute(0, 2, 3, 1)
        absdot = F.conv2d(xc.abs(), wd.abs(), bd.abs(), stride=2, padding=2).permute(0, 2, 3, 1)
        _faithful(got, want, absdot, label, MAX_DIFF_FRAC, ulps=hk.ulps(want, pre=pre))

    def _tran_down(self, i):
        tp, dp = f"block.downtranBlocks.{i - 1}", f"block.downBlocks.{i}"
        tran = (self.w(tp).view(32, -1), self.b(tp), self.slope(tp)) if i > 0 else (None, None, 0.0)
        return tran, (self.w(dp), self.b(dp), self.slope(dp)), tp, dp

    def _down_faithful(self, srcs, i, got, label):
        (_, bt, s_t), (_, bd, s_d), tp, dp = self._tran_down(i)
        wt = self.rw(tp).view(32, -1) if i > 0 else None
        want, absdot, extra = hk.down_faithful(srcs, wt, bt, s_t, self.rw(dp), bd, s_d)
        _faithful(got, want, absdot, label, _MAX_DIFF_FRAC_FUSED, extra=extra)

    def fused(self, inp, label, group):
        i, got = group, self.p.views[LR(group + 1)]
        tran, dn, _, _ = self._tran_down(i)
        hr = torch.stack([inp[HR(j)] for j in range(i + 1)])
        hk.bits_equal(got, hk.fused_down(hr, *tran, *dn), f"{label} vs vsr_test_fused_down")
        self._down_faithful([(_d(hk.from_block(inp[HR(j)])), None) for j in range(i + 1)], i, got, label)

    def updown(self, inp, label, group, up_in):
        i, p = group, self.p
        store = i + 1 < 6                                   # hr[5] is read by no later group
        up = f"block.upBlocks.{i}"
        tran, dn, _, _ = self._tran_down(i)
        hr = torch.empty((i + 1, p.M, 8, p.h + 1, p.w + 1, 64), dtype=torch.bfloat16, device=DEV)
        for j in range(i):
            hr[j].copy_(inp[HR(j)])
        y, hr_after = hk.fused_updown(inp[up_in], hr, store, self.w(up), self.b(up), self.slope(up), *tran, *dn)
        got = p.views[LR(i + 1)]
        hk.bits_equal(got, y, f"{label} lr[{i + 1}] vs vsr_test_fused_updown")
        if store:
            hk.bits_equal(p.views[HR(i)], hr_after[i], f"{label} hr[{i}] vs vsr_test_fused_updown",
                          dims="b,pair,Yb,Xb,el")
            _ring_zero(p.views[HR(i)], f"{label} hr[{i}]")
        xc, wu, bu = _d(inp[up_in]).permute(0, 3, 1, 2), self.rw(up), _d(self.b(up))
        pre_u = F.conv_transpose2d(xc, wu, bu, stride=4, padding=2).permute(0, 2, 3, 1)
        abs_u = F.conv_transpose2d(xc.abs(), wu.abs(), bu.abs(), stride=4, padding=2).permute(0, 2, 3, 1)
        u = self.R.act_packed(pre_u, self.sd, up)
        if store:
            _faithful(hk.from_block(p.views[HR(i)]), u, abs_u, f"{label} hr[{i}]", MAX_DIFF_FRAC,
                      ulps=hk.ulps(u, pre=pre_u))
        self._down_faithful([(_d(hk.from_block(inp[HR(j)])), None) for j in range(i)] + [(u, abs_u)], i, got, label)

    def conv_out(self, inp, label):
        p, sd = self.p, self.sd
        hb, got = inp[HB], p.views[PREMIX]
        hook = hk.conv_out(hb, p.x, p.s, self.w("conv_out"), self.b("conv_out"), sd["sub_mean.bias"],
                           sd["add_mean.bias"])
        if not torch.equal(got.view(torch.int32), hook.view(torch.int32)):
            n = int((got.view(torch.int32) != hook.view(torch.int32)).sum())
            raise AssertionError(f"{label} vs vsr_test_conv_out: {n}/{got.numel()} elements differ")
        hbd = _d(hb).permute(0, 3, 1, 2)
        want = self.R.conv_out(hbd, _d(p.x), sd, p.s)
        tol = 16 * 2.0 ** -24 * hk.conv_out_abs(hbd, p.x, sd, p.s)
        err = (got.double() - want).abs()
        bad = (err > tol).nonzero()
        assert bad.numel() == 0, f"{label}: {bad.shape[0]} pixels outside, first (b,c,y,x) " \
                                 f"{[tuple(i.tolist()) for i in bad[:6]]}"
        print(f"[measure] {label}: worst err/tol {(err / tol).max().item():.3f}")


def _inputs(kind, a):
    return {"conv_in": [], "pw": a.get("srcs", []), "up": [a.get("src")], "down2": [a.get("src")],
            "fused": [HR(j) for j in range(a.get("group", 0) + 1)],
            "updown": [a.get("up_in")] + [HR(j) for j in range(a.get("group", 0))], "conv_out": [HB]}[kind]


def _outputs(kind, a):
    """The buffers a step may write: its output, the fp32 partial slots of the fused kernels, the im2col of conv_in."""
    if kind == "conv_in":
        return [A0, C128]
    if kind == "conv_out":
        return [PREMIX]
    if kind == "fused":
        return [LR(a["group"] + 1), ACC]
    if kind == "updown":
        return [LR(a["group"] + 1), ACC] + ([HR(a["group"])] if a["group"] < 5 else [])
    return [a["out"]]


def _no_stray_writes(plan, before, allowed):
    ws = plan.ent["workspace"]
    diff = ws != before
    for k in allowed:
        off, n = plan.ranges[k]
        diff[off:off + n] = False
    if bool(diff.any()):
        i = int(diff.to(torch.uint8).argmax())
        owner = next((k for k, (o, n) in plan.ranges.items() if o <= i < o + n), "an alignment gap")
        raise AssertionError(f"{int(diff.sum())} bytes written outside its outputs, the first at byte {i} ({owner})")


def _walk(plan, sd, seq, R):
    """Runs the plan's layer list step by step from a workspace of 0xFF bytes; raises LayerMismatch at the first step
    that fails a check.  Returns the number of steps."""
    assert [c for _, cs, _, _ in seq for c in cs] == plan.classes, "layer sequence"
    checks = _Checks(plan, sd, R)
    ws = plan.ent["workspace"]
    ws.fill_(0xFF)
    first = 0
    for label, classes, kind, a in seq:
        inp = {k: plan.views[k].clone() for k in _inputs(kind, a)}
        before = ws.clone()
        hk.run_layers(plan.ent, plan.x, first, len(classes))
        first += len(classes)
        try:
            getattr(checks, kind)(inp, label, **a)
            _no_stray_writes(plan, before, _outputs(kind, a))
        except AssertionError as e:
            raise LayerMismatch(label, str(e)) from None
    assert first == len(plan.classes)
    return len(seq)


_CASES = ([(3, 9, 21, 3, s) for s in (4, 2)] + [(2, hw[0], hw[1], 2, s) for s in (4, 2) for hw in ((1, 1), (13, 1), (1, 17))]
          # several 1x1 tiles per CTA: x4 57,600 LR rows = 450 tiles; x2 the downtran's 115,200 HR rows = 900 tiles
          + [(8, 80, 90, 1, 4), (8, 40, 90, 1, 2)])


@pytest.mark.parametrize("M,h,w,steps,scale", _CASES)
def test_plan_walk(M, h, w, steps, scale):
    """Every layer of the bound plan: hook identity, restatement agreement and no stray writes; the layer sequence is
    the graph's; after the walk the per-map images are the whole forward's, bit for bit."""
    t0 = time.time()
    sd = hk.stack_state(M, h, scale)
    plan = _Plan(sd, M, h, w, steps, scale)
    n = _walk(plan, sd, _plan_steps(scale, steps), sb.Restatement())
    assert torch.equal(plan.views[PREMIX].view(torch.int32), plan.premix.view(torch.int32)), "premix after the walk"
    print(f"[measure] walk M={M} {h}x{w} steps={steps} x{scale}: {n} steps, {len(plan.classes)} layers, "
          f"{time.time() - t0:.1f} s")


# ---- sensitivity -----------------------------------------------------------------------------------------------------
class _HiddenIsX(sb.Restatement):
    """compress_in of the second feedback step reads x twice, as the first does."""

    def __init__(self):
        super().__init__()
        self.calls = 0

    def feedback_block(self, x, last_hidden, sd, num_groups, scale):
        self.calls += 1
        return super().feedback_block(x, x if self.calls == 2 else last_hidden, sd, num_groups, scale)


def _perturbed(kind, sd, seq):
    """(state dict, walk steps, restatement) of the expected side with one deliberate error; the kernels are
    untouched."""
    sd, seq = dict(sd), list(seq)
    if kind == "uptranBlocks.2 given the slope of uptranBlocks.3":
        sd["block.uptranBlocks.2.1.weight"] = sd["block.uptranBlocks.3.1.weight"]
        return sd, seq, sb.Restatement()
    if kind == "compress_in at step 1 fed xfeat twice":
        k = next(n for n, st in enumerate(seq) if st[0] == "step 1 compress_in")
        label, classes, kk, a = seq[k]
        seq[k] = (label, classes, kk, dict(a, srcs=[XFEAT, XFEAT]))
        return sd, seq, _HiddenIsX()
    if kind == "one conv_out tap of one channel x 1.01":
        sd["conv_out.0.weight"] = sd["conv_out.0.weight"].clone()
        sd["conv_out.0.weight"][1, :, 0, 2] *= 1.01
        return sd, seq, sb.Restatement()
    return sd, seq, sb.Restatement(exact_slopes={"block.compress_in"})


_PERTURBATIONS = {"uptranBlocks.2 given the slope of uptranBlocks.3": "step 0 uptranBlocks.2",
                  "compress_in at step 1 fed xfeat twice": "step 1 compress_in",
                  "one conv_out tap of one channel x 1.01": "conv_out",
                  "compress_in's slope left unrounded": "step 0 compress_in"}


@pytest.mark.parametrize("scale", [4, 2])
def test_walk_rejects_a_perturbed_expectation_at_its_layer(scale):
    """Each perturbation of the expected side is reported at exactly the layer it touches.  Whether the whole-stack
    bounds of test_full_stack_against_restatement (same case, same state, same maps) reject the same perturbation of
    the restatement is printed.  Measured on a B200, they reject only compress_in fed xfeat twice (max 10.6 / 42.3 at
    x4 / x2); the other three leave the whole stack within its bounds (max 0.064 to 0.072 at x4, 0.28 to 0.42 at x2, the
    size of the clean divergence)."""
    M, h, w, steps = 3, 9, 21, 2
    sd = hk.stack_state(M, h, scale)
    plan = _Plan(sd, M, h, w, steps, scale)
    b_max, b_rms, b_fused = STACK_BOUNDS[(M, h, w, steps, scale)]
    for kind, layer in _PERTURBATIONS.items():
        psd, seq, R = _perturbed(kind, sd, _plan_steps(scale, steps))
        with pytest.raises(LayerMismatch) as e:
            _walk(plan, psd, seq, R)
        assert e.value.label == layer, (kind, str(e.value)[:2000])
        want_maps = R.forward_maps(_d(plan.x), psd, steps, 6, scale)
        mx, rms = _map_errors(plan.premix.double(), want_maps)
        fused = (plan.frame.double() - sb.fc_fuse(want_maps, psd)).abs().max().item()
        rejected = mx.max().item() > b_max or rms.max().item() > b_rms or fused > b_fused
        print(f"[measure] perturb x{scale} {kind}: walk stops at '{e.value.label}'; whole stack max "
              f"{mx.max().item():.4g} rms {rms.max().item():.4g} fused {fused:.4g}, whole-stack bounds reject: "
              f"{rejected}")
