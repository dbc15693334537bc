"""GPU: the SR conv stack against its BF16-faithful float64 restatement (oracle/srfbn_bf16.py).  The restatement rounds
to BF16 where the kernels round, so only the order of the fp32 accumulations separates the two.

One layer at a time that is tight: conv_in, conv_out (vsr_test_conv_in / vsr_test_conv_out) and the fc fuse agree with
the restatement to an ulp or to the fp32 error bound of their sums, so an error in one border pixel, one tile seam or
one tap is seen.  Through the whole stack it is not: where an fp32 sum lies next to a BF16 rounding boundary (up to
0.6 % of a layer's outputs, measured) the two sides round that element one ulp apart, and 40-odd layers over three
feedback steps carry these flips on.  Measured on a B200, the per-map difference to the restatement is only 1.2 to 1.7
times smaller than to the fp32 oracle (e.g. C2 maps: max 0.108, RMS 0.0145 on the 0..255 scale).  The whole-stack
bounds below are still set per case at about 4x the measured values -- an order of magnitude under the fp32 criteria
of test_srfbn_gpu.py -- and reject a border or padding error of the conv_in / skip kind; errors as small as one
conv_out tap off by 1 % or one PReLU slope left unrounded are rejected by the single-layer checks instead.

At the benchmark's sizes a whole-map max and RMS cannot see an error confined to a few rows or one corner of a map,
so there every region of a map -- its border bands and its tiles of 32 x 32 LR blocks -- is held to a bound too."""
import gc
import math
import time

import pytest
import torch
import torch.nn.functional as F

from oracle import srfbn_bf16 as sb
from oracle import srfbn_oracle as so
from tests import srfbn_hooks as hk
from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
# of one layer's BF16 outputs that may differ at all from the restatement (hk.faithful_bf16): conv_in measured 0.0006 %
# on a B200; the one-GEMM layers of test_srfbn_gpu.py up to 0.044 %
MAX_DIFF_FRAC = 0.002


def _d(t):
    return t.to(DEV, torch.float64)


# ---- conv_in ------------------------------------------------------------------------------------------------------
# (1, 160, 250): 40000 rows = 313 tiles of 128 on 296 CTAs, so some CTAs walk two tiles
@pytest.mark.parametrize("B,h,w,slope", [(1, 1, 1, 0.2), (3, 1, 17, 0.2), (1, 13, 1, 0.2), (3, 5, 7, 0.2),
                                         (1, 19, 33, 0.2), (3, 19, 33, -0.3), (1, 5, 7, 1.7), (1, 160, 250, 0.2)])
def test_conv_in_against_restatement(B, h, w, slope):
    g = torch.Generator().manual_seed(B * 1000 + h * 37 + w)
    x = torch.rand((B, 3, h, w), generator=g) * 255
    sd = {"sub_mean.bias": -255.0 * torch.tensor(so.RGB_MEAN),
          "conv_in.0.weight": torch.randn((128, 3, 3, 3), generator=g) / math.sqrt(27),
          "conv_in.0.bias": torch.randn(128, generator=g),
          "conv_in.1.weight": torch.tensor([slope])}
    got = hk.conv_in(x.to(DEV), sd["conv_in.0.weight"], sd["conv_in.0.bias"], slope, sd["sub_mean.bias"])
    R = sb.Restatement()
    want = R.conv_in(_d(x), sd).permute(0, 2, 3, 1)
    xs = R.rb(_d(x) + _d(sd["sub_mean.bias"]).view(1, 3, 1, 1))
    absdot = F.conv2d(xs.abs(), R.weight(sd, "conv_in", DEV).abs(), _d(sd["conv_in.0.bias"]).abs(), padding=1)
    hk.faithful_bf16(got, want, absdot.permute(0, 2, 3, 1), f"conv_in B={B} {h}x{w} slope={slope}",
                     max_frac=MAX_DIFF_FRAC, ulps=torch.where(want < 0, 2.0, 1.0))


# ---- conv_out -----------------------------------------------------------------------------------------------------
# HR width W = s*w with W % 14 in {0, 2, 12} and height H = s*h with H % 6 in {0, 2, 4} (14 x 6 output tiles); LR 1 x 1,
# 1 x w and h x 1 put the skip's clamps on both sides; B up to 5 walks the TMA batch dimension and the skip's image
# index; (2, 30, 40, 4) and (4, 60, 80, 2) have 480 and 960 tiles on 444 CTAs.
_CONV_OUT_CASES = [(1, 1, 1, 4), (1, 1, 7, 4), (3, 3, 1, 4), (1, 2, 10, 4), (5, 3, 4, 4), (3, 13, 17, 4),
                   (2, 30, 40, 4), (1, 1, 1, 2), (1, 2, 7, 2), (3, 3, 1, 2), (5, 1, 6, 2), (3, 13, 17, 2),
                   (4, 60, 80, 2)]


def _conv_out_operands(B, h, w, scale, seed):
    g = torch.Generator().manual_seed(seed)
    hb = torch.randn((B, scale * h, scale * w, 32), generator=g).to(torch.bfloat16)
    x = torch.rand((B, 3, h, w), generator=g) * 255
    sd = {"sub_mean.bias": torch.tensor([-114.4, -111.5, -103.0]),     # three distinct mean shifts each way
          "add_mean.bias": torch.tensor([114.4, 111.5, 103.0]) + torch.randn(3, generator=g),
          "conv_out.0.weight": torch.randn((3, 32, 3, 3), generator=g) / math.sqrt(288) * 8,
          "conv_out.0.bias": torch.randn(3, generator=g)}
    return hb, x, sd


@pytest.mark.parametrize("B,h,w,scale", _CONV_OUT_CASES)
def test_conv_out_against_fp64(B, h, w, scale):
    """conv_out's fp32 output against float64 on the same BF16 operands: |got - want| <= 16 * 2^-24 * sum |terms| per
    pixel (the fp32 partial sums and the fp32 skip); output poisoned with NaN, guard bands intact (hk.conv_out)."""
    hb, x, sd = _conv_out_operands(B, h, w, scale, seed=B * 100 + h * 10 + w + scale)
    got = hk.conv_out(hb.to(DEV), x.to(DEV), scale, sd["conv_out.0.weight"], sd["conv_out.0.bias"],
                      sd["sub_mean.bias"], sd["add_mean.bias"]).double()
    assert torch.isfinite(got).all()
    hbd = _d(hb).permute(0, 3, 1, 2)
    want = sb.Restatement().conv_out(hbd, _d(x), sd, scale)
    tol = 16 * 2.0 ** -24 * hk.conv_out_abs(hbd, x, sd, scale)
    err = (got - want).abs()
    bad = (err > tol).nonzero()
    assert bad.numel() == 0, f"{bad.shape[0]} pixels outside, first (b,c,y,x) {[tuple(i.tolist()) for i in bad[:6]]}"
    print(f"[measure] conv_out B={B} {h}x{w} x{scale}: max err {err.max().item():.3g} worst err/tol "
          f"{(err / tol).max().item():.3f}")


# ---- fc fuse ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [1, 2, 3, 5, 8, 20, 63, 64])
def test_fc_fuse_teacher_forced(M):
    """The fused frame against an fp64 fc over the stack's own per-map images: within the error bound of the kernel's
    fp32 FMA chains (hid_j: M + 1 terms, o: 33 terms)."""
    h, w = 3, 5
    sd = so.init_state_dict(num_maps=M, seed=M, gain=2.3)
    sd["fc.2.weight"] = sd["fc.2.weight"].abs()          # a frame the final ReLU does not zero: the check is not blind
    mod = SRProjectionModule(num_maps=M)
    mod.load_state_dict(sd)
    x = (torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(M + 1)) * 255).to(DEV)
    maps = mod.premix(x).double()
    got = mod(x).double()
    want = sb.fc_fuse(maps, sd)
    bound = hk.fc_fuse_bound(maps, sd)
    err = (got - want).abs()
    assert (err <= bound).all(), \
        f"M={M}: max err {err.max().item():.3g}, worst err/bound {(err / bound).max().item():.3f}"
    assert want.abs().mean().item() > 1.0                 # the fc carries signal
    print(f"[measure] fc_fuse M={M}: max err {err.max().item():.3g} worst err/bound {(err / bound).max().item():.3f}")


def test_fc_fuse_u8_rounds_half_to_even():
    """vsr_srfbn_fuse_band with M = 1 and an identity fc (o = relu(map)): maps at k + 0.5 for k = -1..255, at +-1e30 and
    at the fp32 neighbours of 0.5 give the u8 frame round-half-to-even(clamp(o, 0, 255)) exactly and the fp32 frame
    relu(map) exactly."""
    from video_super_resolution_b200 import _lib
    h, w, s = 3, 8, 4
    sd = so.init_state_dict(num_maps=1, seed=0)
    sd["fc.0.weight"] = torch.zeros(32, 1)
    sd["fc.0.weight"][0, 0] = 1.0
    sd["fc.0.bias"] = torch.zeros(32)
    sd["fc.2.weight"] = torch.zeros(1, 32)
    sd["fc.2.weight"][0, 0] = 1.0
    sd["fc.2.bias"] = torch.zeros(1)
    mod = SRProjectionModule(num_maps=1)
    mod.load_state_dict(sd)
    ent = mod._plan_for(1, h, w, torch.device(DEV))
    rows, W = s * h, s * w
    f32 = torch.float32

    def nb(v, to):        # the fp32 neighbour of v towards `to`
        return torch.nextafter(torch.tensor(v, dtype=f32), torch.tensor(to, dtype=f32))

    special = torch.cat([torch.arange(-1, 256, dtype=f32) + 0.5,
                         torch.tensor([1e30, -1e30, 255.0, 256.0, -0.0], dtype=f32),
                         torch.stack([nb(0.5, 0.0), nb(0.5, 1.0), nb(254.5, 300.0), nb(255.5, 0.0), nb(1.5, 0.0)])])
    vals = torch.rand(3 * rows * W, generator=torch.Generator().manual_seed(3)) * 320 - 20
    vals[:special.numel()] = special
    maps = vals.view(1, 3, rows, W).to(DEV)
    y = torch.full((3, rows, W), float("nan"), device=DEV)
    y8 = torch.zeros((rows, W, 3), dtype=torch.uint8, device=DEV)
    _lib.check(_lib.lib().vsr_srfbn_fuse_band(ent["plan"], maps.data_ptr(), rows, y.data_ptr(), y8.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream), "fuse_band")
    m32 = maps[0].cpu()
    assert torch.equal(y.cpu(), torch.relu(m32))
    want8 = torch.round(m32.double().clamp(0, 255)).to(torch.uint8).permute(1, 2, 0)
    bad = (y8.cpu() != want8).nonzero()
    assert bad.numel() == 0, \
        [(m32.permute(1, 2, 0)[tuple(i)].item(), y8.cpu()[tuple(i)].item()) for i in bad[:8].tolist()]


# ---- the whole stack ----------------------------------------------------------------------------------------------
_STACK_CASES = [(8, 16, 16, 3, 4), (3, 9, 21, 2, 4), (20, 24, 40, 3, 4), (8, 16, 16, 3, 2), (3, 9, 21, 2, 2),
                (14, 24, 40, 3, 2), (2, 37, 19, 1, 2), (2, 1, 1, 2, 4), (2, 1, 17, 2, 4), (2, 13, 1, 2, 4),
                (2, 1, 1, 2, 2), (2, 1, 17, 2, 2), (2, 13, 1, 2, 2)]
# Per case: (max-abs, RMS) over the maps of |premix - restatement|, and max-abs of |fused frame - fc(restatement)|, on
# the 0..255 scale.  About 4x the values measured on one NVIDIA B200 (1000 W power limit), given in the comments as
# (max, RMS, fused); against the fp32 oracle the same cases measured 1.2-1.7x larger (x2 1 x 1: 350x -- no flips there).
STACK_BOUNDS = {
    (8, 16, 16, 3, 4): (0.3, 0.053, 0.11),            # 0.0729, 0.0131, 0.0265
    (3, 9, 21, 2, 4): (0.26, 0.05, 0.13),             # 0.0636, 0.0125, 0.0319
    (20, 24, 40, 3, 4): (0.38, 0.059, 0.1),           # 0.0949, 0.0147, 0.0252
    (8, 16, 16, 3, 2): (1.4, 0.34, 0.42),             # 0.341, 0.0837, 0.104
    (3, 9, 21, 2, 2): (1.2, 0.27, 0.35),              # 0.289, 0.0678, 0.0873
    (14, 24, 40, 3, 2): (2.0, 0.39, 0.53),            # 0.500, 0.0974, 0.133
    (2, 37, 19, 1, 2): (1.5, 0.3, 0.54),              # 0.362, 0.0741, 0.135
    (2, 1, 1, 2, 4): (0.0082, 0.0029, 0.0026),        # 0.00205, 0.000712, 0.000654
    (2, 1, 17, 2, 4): (0.056, 0.012, 0.0076),         # 0.0140, 0.00306, 0.00190
    (2, 13, 1, 2, 4): (0.051, 0.012, 0.022),          # 0.0126, 0.00307, 0.00543
    (2, 1, 1, 2, 2): (4.3e-5, 2.3e-5, 6.7e-5),        # 1.08e-5, 5.78e-6, 1.67e-5
    (2, 1, 17, 2, 2): (0.058, 0.023, 0.024),          # 0.0144, 0.00569, 0.00608
    (2, 13, 1, 2, 2): (0.075, 0.027, 0.038),          # 0.0186, 0.00679, 0.00948
}
C2_BOUNDS = (0.43, 0.058)                             # maps 0 and 19: 0.108, 0.0145 (restatement 1.0 s)


def _stack_run(M, h, w, steps, scale):
    sd = hk.stack_state(M, h, scale)
    mod = SRProjectionModule(num_steps=steps, num_maps=M, upscale_factor=scale)
    mod.load_state_dict(sd)
    x = torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(5)) * 255
    got_maps = mod.premix(x.to(DEV)).double()
    got = mod(x.to(DEV)).double()
    assert torch.isfinite(got_maps).all() and torch.isfinite(got).all()
    return sd, x, got_maps, got


def _map_errors(got_maps, want_maps):
    d = (got_maps - want_maps).flatten(1)
    return d.abs().max(dim=1).values, d.pow(2).mean(dim=1).sqrt()


@pytest.mark.parametrize("M,h,w,steps,scale", _STACK_CASES)
def test_full_stack_against_restatement(M, h, w, steps, scale):
    sd, x, got_maps, got = _stack_run(M, h, w, steps, scale)
    want_maps = sb.forward_maps(_d(x), sd, num_steps=steps, upscale=scale)
    skip = F.interpolate(_d(x), scale_factor=scale, mode="bilinear", align_corners=False)
    assert (want_maps - skip).abs().mean().item() > 0.05          # the conv branch carries signal: not blind
    mx, rms = _map_errors(got_maps, want_maps)
    want = sb.fc_fuse(want_maps, sd)
    fused = (got - want).abs().max().item()
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):      # a true fp32 oracle, not TF32
        f32_maps = so.forward_maps(x.to(DEV), {k: v.to(DEV) for k, v in sd.items()}, num_steps=steps,
                                   upscale=scale).double()
    mx32, rms32 = _map_errors(got_maps, f32_maps)
    print(f"[measure] stack M={M} {h}x{w} steps={steps} x{scale}: restatement max {mx.max().item():.4g} rms "
          f"{rms.max().item():.4g} fused {fused:.4g}; fp32 oracle max {mx32.max().item():.4g} "
          f"rms {rms32.max().item():.4g}")
    b_max, b_rms, b_fused = STACK_BOUNDS[(M, h, w, steps, scale)]
    assert mx.max().item() <= b_max and rms.max().item() <= b_rms and fused <= b_fused, \
        (mx.max().item(), rms.max().item(), fused)


def test_full_stack_c2_maps_against_restatement():
    """C2: M = 20 maps of 270 x 480, x4.  The maps are independent until the fc fuse, so maps 0 and 19 are restated
    (CUDA float64) and checked with the same per-map bounds."""
    M, h, w = 20, 270, 480
    sd = so.init_state_dict(num_maps=M, seed=2, gain=2.3)
    mod = SRProjectionModule(num_maps=M)
    mod.load_state_dict(sd)
    x = torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(4)) * 255
    got_maps = mod.premix(x.to(DEV)).double()[[0, M - 1]]
    t0 = time.time()
    want_maps = sb.forward_maps(_d(x[[0, M - 1]]), sd)
    torch.cuda.synchronize()
    mx, rms = _map_errors(got_maps, want_maps)
    print(f"[measure] stack C2 maps 0,19: max {mx.max().item():.4g} rms {rms.max().item():.4g} "
          f"(restatement {time.time() - t0:.1f} s)")
    assert mx.max().item() <= C2_BOUNDS[0] and rms.max().item() <= C2_BOUNDS[1], (mx.tolist(), rms.tolist())


# ---- the stack at the benchmark's sizes ---------------------------------------------------------------------------
# hk.FULL_SIZE_PLANS cases, their restated maps and bounds on |premix - restatement| (0..255 scale): whole-map max-abs,
# which every region's max-abs must meet too; whole-map RMS; every region's RMS (hk.region_errors: the 2*scale-pixel
# border bands and the tiles over 32 x 32 LR blocks); and, where every map is restated, max-abs of |fused frame -
# fc(restatement)|.  About 4x the values measured on one NVIDIA B200 (1000 W power limit), given in the comments as
# (max, RMS, region RMS, fused).  In the same run the restatement, one map at a time, peaked at 9.8 (C2), 20.6 (C5) and
# 43.0 GiB (C4) allocated, and in the whole suite the three cases took 1.5, 8.0 and 8.5 s.
FULL_SIZE_MAPS = {"C2": (0, 19), "C5": tuple(range(8)), "C4": (0, 13)}
FULL_SIZE_BOUNDS = {
    "C2": (0.58, 0.086, 0.089, None),                 # maps 0, 19: 0.1435, 0.02135, 0.02209
    "C5": (0.33, 0.046, 0.048, 0.068),                # maps 0..7: 0.08289, 0.01135, 0.01183, 0.01699
    "C4": (2.3, 0.37, 0.39, None),                    # maps 0, 13: 0.565, 0.092, 0.09638
}


def _teacher_forced_fuse(maps, got, sd, what):
    """The fused frame got (1,3,H,W) against sb.fc_fuse over the stack's own per-map images maps (M,3,H,W), within
    hk.fc_fuse_bound, one colour channel at a time (C4's float64 hidden layer is 2 GB per channel).  Returns the worst
    err / bound."""
    worst = 0.0
    for c in range(3):
        m = maps[:, c:c + 1]
        want = sb.fc_fuse(m, sd)
        err = (got[:, c:c + 1].double() - want).abs()
        ratio = (err / hk.fc_fuse_bound(m, sd)).max().item()
        assert ratio <= 1.0, f"{what}: channel {c} max err {err.max().item():.3g}, worst err/bound {ratio:.3f}"
        assert want.abs().mean().item() > 1.0                 # the fc carries signal
        worst = max(worst, ratio)
    return worst


def _full_size_run(name):
    """One plan forward of case `name` on stack_state weights and fp32 frames: (state dict, x, premix, fused frame)."""
    M, h, w, scale, _, _ = hk.FULL_SIZE_PLANS[name]
    sd = hk.stack_state(M, h, scale)
    mod = SRProjectionModule(num_maps=M, upscale_factor=scale)
    mod.load_state_dict(sd)
    x = (torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(4)) * 255).to(DEV)
    premix = mod.premix(x)
    got = mod(x)
    assert torch.isfinite(premix).all() and torch.isfinite(got).all()
    del mod                                               # the plan's workspace: 89 GB at C4
    gc.collect()
    torch.cuda.empty_cache()
    return sd, x, premix, got


@pytest.mark.parametrize("name", ["C2", "C5", "C4"])
def test_full_size_maps_against_restatement(name):
    """The conv stack at the benchmark's sizes, where 32-bit offsets, TMA coordinates and the last rows of the last map
    are exercised: C2 (M = 20, 270 x 480, x4; the HR ring over 2^31 bytes), C5 (M = 8, 360 x 720, x4) and C4 (M = 14,
    1080 x 1920, x2, uncapped as bench.py runs it; buffers over 2^31 BF16 elements).  The maps are independent until
    the fc fuse, so the first and last maps are restated (all of them at C5), one at a time in CUDA float64, and held to
    whole-map and per-region bounds; the fused frame is checked teacher-forced over all M maps, and at C5 also against
    the fc over the restated maps."""
    M, h, w, scale, _, _ = hk.FULL_SIZE_PLANS[name]
    maps = FULL_SIZE_MAPS[name]
    b_max, b_rms, b_region_rms, b_fused = FULL_SIZE_BOUNDS[name]
    gc.collect()
    torch.cuda.empty_cache()
    t0 = time.time()
    sd, x, premix, got = _full_size_run(name)
    tf = _teacher_forced_fuse(premix, got, sd, f"{name} teacher-forced fc fuse")
    got_maps = premix[list(maps)].clone()
    del premix
    torch.cuda.empty_cache()
    t1 = time.time()
    torch.cuda.reset_peak_memory_stats()
    held = torch.cuda.memory_allocated()
    mx, rms, region_mx, region_rms, fails, wants = [], [], 0.0, 0.0, [], []
    for i, m in enumerate(maps):
        want = sb.forward_maps(x[m:m + 1], sd, upscale=scale)
        if i == 0:                                        # the conv branch carries signal: not blind
            skip = F.interpolate(x[m:m + 1].double(), scale_factor=scale, mode="bilinear", align_corners=False)
            assert (want - skip).abs().mean().item() > 0.05
            del skip
        d = got_maps[i:i + 1].double() - want
        mx.append(d.abs().max().item())
        rms.append(d.square().mean().sqrt().item())
        del d
        regs, rmx, rrms = hk.region_errors(got_maps[i:i + 1], want, scale)
        region_mx, region_rms = max(region_mx, rmx.max().item()), max(region_rms, rrms.max().item())
        fails += hk.region_failures(regs, rmx, rrms, b_max, b_region_rms, [m])
        if b_fused is not None:
            wants.append(want)
        del want
    torch.cuda.synchronize()
    t2 = time.time()
    peak = torch.cuda.max_memory_allocated()
    fused = None
    if b_fused is not None:
        fused = (got.double() - sb.fc_fuse(torch.cat(wants), sd)).abs().max().item()
    print(f"[measure] full-size {name} maps {maps[0]}..{maps[-1]}: max {max(mx):.4g} rms {max(rms):.4g} region max "
          f"{region_mx:.4g} region rms {region_rms:.4g} fused {fused if fused is None else f'{fused:.4g}'}; "
          f"teacher-forced fc worst err/bound {tf:.3f}; forward + fc check {t1 - t0:.1f} s, restatement "
          f"{t2 - t1:.1f} s, restatement peak {peak / 2**30:.1f} GiB allocated ({(peak - held) / 2**30:.1f} GiB over "
          f"the {held / 2**30:.2f} GiB held)")
    assert max(mx) <= b_max and max(rms) <= b_rms, (name, mx, rms)
    assert not fails, f"{name}: {len(fails)} regions outside: " + "; ".join(fails[:12])
    if b_fused is not None:
        assert fused <= b_fused, (name, fused)


# C5's last map restated with its input raised by this much (0..255 scale) in the bottom-right 8 x 8 LR pixels
CORNER_DELTA = 0.1


def test_region_bounds_see_an_error_in_the_last_corner():
    """A deliberate error on the expected side: C5's last map restated from an input raised by CORNER_DELTA in its
    bottom-right 8 x 8 LR pixels (the kernels are untouched) -- an error where the addresses are highest, in 0.025 % of
    the map's pixels.  Some region must exceed the C5 bounds, and only regions within the x4 receptive field of that
    corner (48 LR px) may.  Measured on one NVIDIA B200 (1000 W power limit), whole map / corner tile (LR y 352:360
    x 704:720):
      clean           max 0.0829  RMS 0.0114    corner tile RMS 0.0115
      +0.05           max 0.110   RMS 0.0114    0.0370
      +0.1 (used)     max 0.160   RMS 0.0114    0.0706   -> whole-map bounds (0.33, 0.046) pass it; the region RMS
                                                            bound 0.048 rejects the corner tile, and no other region
      +0.2            max 0.269   RMS 0.0118    0.139
      +0.3            max 0.366   RMS 0.0122    0.208    -> the whole-map max rejects it from here on
    Every region outside the receptive field stays at max 0.0829, RMS 0.0117 at every size of the change."""
    name = "C5"
    M, h, w, scale, _, _ = hk.FULL_SIZE_PLANS[name]
    b_max, b_rms, b_region_rms, _ = FULL_SIZE_BOUNDS[name]
    gc.collect()
    torch.cuda.empty_cache()
    sd, x, premix, _ = _full_size_run(name)
    got = premix[M - 1:M].clone()
    del premix
    xp = x[M - 1:M].clone()
    xp[:, :, -8:, -8:] += CORNER_DELTA
    want = sb.forward_maps(xp, sd, upscale=scale)
    d = got.double() - want
    mx, rms = d.abs().max().item(), d.square().mean().sqrt().item()
    regs, rmx, rrms = hk.region_errors(got, want, scale)
    flagged = [regs[r] for r in ((rmx[0] > b_max) | (rrms[0] > b_region_rms)).nonzero().flatten().tolist()]
    H, W, reach = scale * h, scale * w, scale * (8 + 48)
    far = [r[0] for r in flagged if r[2] <= H - reach or r[4] <= W - reach]
    print(f"[measure] corner +{CORNER_DELTA}: whole-map max {mx:.4g} rms {rms:.4g}, rejected by the whole-map bounds "
          f"alone: {mx > b_max or rms > b_rms}; region max {rmx.max().item():.4g} rms {rrms.max().item():.4g}, "
          f"flagged {[r[0] for r in flagged]}")
    assert flagged, "the region bounds miss an error in the last map's bottom-right corner"
    assert not far, f"regions outside the corner's receptive field flagged: {far}"


# ---- sensitivity --------------------------------------------------------------------------------------------------
def _perturbed(sd, kind):
    """(restatement options, state dict) of one deliberate error in the RESTATEMENT (the kernels are untouched)."""
    if kind == "conv_in pads x, not sub_mean(x)":
        return {"pad_unshifted": True}, sd
    if kind == "skip zero-extended, not clamped":
        return {"skip_zero_ext": True}, sd
    if kind == "one conv_out tap of one channel x 1.01":
        sd = dict(sd)
        sd["conv_out.0.weight"] = sd["conv_out.0.weight"].clone()
        sd["conv_out.0.weight"][1, :, 0, 2] *= 1.01
        return {}, sd
    return {"exact_slopes": {"block.compress_in"}}, sd


_PERTURBATIONS = ["conv_in pads x, not sub_mean(x)", "skip zero-extended, not clamped",
                  "one conv_out tap of one channel x 1.01", "one layer's PReLU slope unrounded"]


def _psnr(a, b):
    return 10 * math.log10(255.0 ** 2 / max(((a - b) ** 2).mean().item(), 1e-20))


def _fp32_criteria(got_maps, want_maps, got, want):
    """The three criteria of test_full_stack_against_oracle, with want in the place of the fp32 oracle."""
    wm, gm = want_maps.cpu(), got_maps.cpu()
    noise = torch.randn(wm.shape, generator=torch.Generator().manual_seed(6), dtype=torch.float64) * 4.5
    delta = abs(_psnr(gm, wm + noise) - _psnr(wm, wm + noise))
    fe = (got - want).abs()
    fused_ok = fe.max().item() <= 0.02 * (want.abs().mean().item() + 1.0) + 0.05 * fe.mean().item() + 0.5
    return _psnr(gm, wm) > 50.0, delta <= 0.05, fused_ok


@pytest.mark.parametrize("scale", [4, 2])
@pytest.mark.parametrize("kind", _PERTURBATIONS)
def test_bounds_reject_a_perturbed_restatement(kind, scale):
    """Each perturbation of the restatement is rejected.  Measured on a B200 (case (3, 9, 21, 2)), against the fp32
    criteria of test_full_stack_against_oracle (per-map PSNR > 50 dB / PSNR delta <= 0.05 dB / fused max err):
      conv_in pads x          x4: passes / fails / passes   x2: fails all three     -> whole-stack bounds: rejected
      skip zero-extended      x4, x2: fail all three                                -> whole-stack bounds: rejected
      conv_out tap x 1.01     x4, x2: pass all three; whole-stack difference 0.072 / 0.42 max, the size of the clean
                              divergence -> rejected by the conv_out layer bound
      PReLU slope unrounded   x4, x2: pass all three; whole-stack 0.064 / 0.28 max, the same -> rejected by the
                              faithful single-layer bound."""
    M, h, w, steps = 3, 9, 21, 2
    sd, x, got_maps, got = _stack_run(M, h, w, steps, scale)
    opts, psd = _perturbed(sd, kind)
    want_maps = sb.forward_maps(_d(x), psd, num_steps=steps, upscale=scale, **opts)
    mx, rms = _map_errors(got_maps, want_maps)
    want = sb.fc_fuse(want_maps, psd)
    fused = (got - want).abs().max().item()
    b_max, b_rms, b_fused = STACK_BOUNDS[(M, h, w, steps, scale)]
    rejected = mx.max().item() > b_max or rms.max().item() > b_rms or fused > b_fused
    print(f"[measure] perturb x{scale} {kind}: max {mx.max().item():.4g} rms {rms.max().item():.4g} fused {fused:.4g} "
          f"whole-stack rejected={rejected}; fp32 criteria pass (psnr, delta, fused) = "
          f"{_fp32_criteria(got_maps, want_maps, got, want)}")
    if kind in _PERTURBATIONS[:2]:
        assert rejected, (kind, mx.max().item(), rms.max().item(), fused)
    elif kind == _PERTURBATIONS[2]:       # the conv_out layer on its own, against the perturbed restatement
        hb, xl, lsd = _conv_out_operands(2, 13, 17, scale, seed=scale)
        ysd = dict(lsd, **{"conv_out.0.weight": lsd["conv_out.0.weight"].clone()})
        ysd["conv_out.0.weight"][1, :, 0, 2] *= 1.01
        got_l = hk.conv_out(hb.to(DEV), xl.to(DEV), scale, lsd["conv_out.0.weight"], lsd["conv_out.0.bias"],
                            lsd["sub_mean.bias"], lsd["add_mean.bias"]).double()
        hbd = _d(hb).permute(0, 3, 1, 2)
        tol = 16 * 2.0 ** -24 * hk.conv_out_abs(hbd, xl, lsd, scale)
        assert ((got_l - sb.Restatement().conv_out(hbd, _d(xl), ysd, scale)).abs() > tol).any()
    else:                                 # one layer at slope -0.2 against the restatement with the fp32 slope
        g = torch.Generator().manual_seed(scale)
        xb = torch.randn((4096, 64), generator=g).to(torch.bfloat16)
        wl = torch.randn((32, 64), generator=g).to(torch.bfloat16).float() / 8
        bl = torch.randn(32, generator=g) * 0.1
        got_l = hk.pointwise(xb.to(DEV), wl, bl, -0.2)
        pre = _d(xb) @ _d(wl).t() + _d(bl)
        s32 = float(torch.tensor(-0.2, dtype=torch.float32))
        want_l = sb.prelu_packed(sb.round_bf16(pre), s32, s32)          # slope NOT rounded to BF16
        with pytest.raises(AssertionError, match="outside the faithful bound|differ"):
            hk.faithful_bf16(got_l, want_l, _d(xb).abs() @ _d(wl).abs().t() + _d(bl).abs(), "unrounded slope",
                             max_frac=MAX_DIFF_FRAC, ulps=torch.where(want_l < 0, 2.0, 1.0))
