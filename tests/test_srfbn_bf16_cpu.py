"""CPU checks of the BF16-faithful restatement (oracle/srfbn_bf16.py): without rounding it is the float64 oracle, its
packed-BF16 PReLU is exact over every finite BF16 input, and its rounding helper is the weight packer's f2bf bit for
bit."""
import ctypes

import pytest
import torch

from oracle import srfbn_bf16 as sb
from oracle import srfbn_oracle as so


@pytest.mark.parametrize("scale", [4, 2])
@pytest.mark.parametrize("M,h,w,steps", [(2, 5, 7, 2), (1, 3, 4, 1)])
def test_restatement_without_rounding_is_the_oracle(scale, M, h, w, steps):
    sd = so.init_state_dict(num_maps=M, seed=scale + h, gain=2.3, upscale=scale)
    gs = torch.Generator().manual_seed(7)
    for k in sd:                        # distinct slopes, all three packed-PReLU forms
        if k.endswith(".1.weight"):
            sd[k] = torch.rand(1, generator=gs) * 0.4 + 0.05
    sd["feat_in.1.weight"] = torch.tensor([1.3])
    sd["block.compress_in.1.weight"] = torch.tensor([-0.2])
    x = torch.rand((M, 3, h, w), generator=torch.Generator().manual_seed(3)) * 255
    want = so.forward_maps(x, sd, num_steps=steps, upscale=scale).double()
    got = sb.forward_maps(x, sd, num_steps=steps, upscale=scale, rounding=False)
    assert got.dtype == torch.float64 and got.shape == want.shape
    err = (got - want).abs().max().item()
    assert err <= 1e-6 * (want.abs().max().item() + 1.0) * 64, err    # fp32 oracle against float64
    # with rounding the restatement departs by BF16 drift, not by more
    rounded = sb.forward_maps(x, sd, num_steps=steps, upscale=scale)
    drift = (rounded - want).abs().max().item()
    assert 0 < drift < 3.0, drift


def _finite_bf16():
    bits = torch.arange(0, 1 << 16, dtype=torch.int64)
    v = sb.bits_to_float(bits)
    return v[torch.isfinite(v)]


@pytest.mark.parametrize("slope", [0.0, 1.0, 0.2, 1.7, -0.3, 0.25, 3.0, -1.5])
def test_packed_prelu_over_every_finite_bf16(slope):
    """igemm.cuh prelu_pack in all three forms, on every finite BF16 x: forms max / min against torch's CPU bf16
    arithmetic (bf16 * bf16 is exact in fp32, then rounded once), the general form against the exact float64 value
    rounded once; and all forms agree with x >= 0 ? x : bf16(x * s_b)."""
    x = _finite_bf16()
    s32 = float(torch.tensor(slope, dtype=torch.float32))
    s_b = float(sb.round_bf16(torch.tensor(s32)))
    got = sb.prelu_packed(x, s32, s_b)
    xb = x.to(torch.bfloat16)
    sbt = torch.tensor(s_b, dtype=torch.bfloat16)
    if 0.0 <= s32 <= 1.0:
        want = torch.maximum(xb, xb * sbt).double()
    elif s32 > 1.0:
        want = torch.minimum(xb, xb * sbt).double()
    else:
        want = sb.round_bf16(s_b * torch.clamp(x, max=0.0) + torch.clamp(x, min=0.0))
        assert torch.equal(want, (torch.clamp(xb, max=0) * sbt + torch.clamp(xb, min=0)).double())
    assert torch.equal(got, want), slope
    assert torch.equal(got, torch.where(x >= 0, x, sb.round_bf16(x * s_b)))
    assert torch.equal(sb.round_bf16(got), got)                  # a BF16 value


def _f2bf_of_library(values):
    """The library's own f2bf: vsr_srfbn_pack_weights writes conv_in's weights first, [128][32] with k = c*9+ky*3+kx <
    27 taken from the (128,3,3,3) weight; 3456 values per call."""
    from video_super_resolution_b200 import _lib
    from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
    L = _lib.lib()
    mod = SRProjectionModule(num_maps=1)
    cfg = _lib.SrfbnConfig(1, 4, 4, 1, 6, 32, 4)
    plan = ctypes.c_void_p()
    _lib.check(L.vsr_srfbn_plan_create(ctypes.byref(cfg), ctypes.byref(plan)), "plan_create")
    try:
        host = torch.zeros(int(L.vsr_srfbn_weight_bytes(plan)), dtype=torch.uint8)
        out = []
        n = 128 * 27
        for i in range(0, values.numel(), n):
            chunk = torch.zeros(n, dtype=torch.float32)
            part = values[i:i + n]
            chunk[:part.numel()] = part
            with torch.no_grad():
                mod.conv_in[0].weight.copy_(chunk.view(128, 3, 3, 3))
            W, keep = mod._weights_struct()
            _lib.check(L.vsr_srfbn_pack_weights(plan, ctypes.byref(W), host.data_ptr()), "pack_weights")
            packed = host[:128 * 32 * 2].view(torch.int16).view(128, 32)[:, :27].reshape(-1)
            out.append(packed[:part.numel()].to(torch.int64) & 0xFFFF)
            del keep
        return torch.cat(out)
    finally:
        L.vsr_srfbn_plan_destroy(plan)


def test_round_bf16_is_the_packers_f2bf():
    """Every upper half-word with low halves that make ties (0x8000, even and odd upper halves), values just either side
    of a tie, exact BF16 values, and the largest: NaN payloads of both signs, infinities, subnormals, the overflow to
    infinity of the largest finite floats."""
    upper = torch.arange(0, 1 << 16, dtype=torch.int64)
    lows = torch.tensor([0x0000, 0x0001, 0x7FFF, 0x8000, 0x8001, 0xFFFF], dtype=torch.int64)
    u = ((upper.view(-1, 1) << 16) | lows.view(1, -1)).reshape(-1)
    f = ((u ^ 0x80000000) - 0x80000000).to(torch.int32).view(torch.float32)
    want = _f2bf_of_library(f)
    got = sb.f2bf_bits(f)
    bad = (got != want).nonzero().view(-1)
    assert bad.numel() == 0, [(hex(int(u[i])), hex(int(got[i])), hex(int(want[i]))) for i in bad[:8]]
    # the cases the test is meant to reach are present
    assert bool(torch.isnan(f).any()) and bool(torch.isinf(f).any())
    assert int(((u & 0x7F800000) == 0).sum()) > 0                     # subnormals
    assert int(got[(u == 0x7F7FFFFF).nonzero().view(-1)]) == 0x7F80    # largest finite float rounds to inf
