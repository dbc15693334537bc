"""BF16-faithful float64 restatement of the SR conv stack (TEST INFRASTRUCTURE ONLY, like srfbn_oracle.py).

It follows srfbn_oracle.forward_maps layer for layer, with the same state-dict names and geometry, computes in float64
on the device of its input, and rounds to BF16 exactly where the kernels of libvsr_b200.so round.  Only the order of
the fp32 accumulations then separates it from the GPU stack, so a whole-stack comparison against it can be far
tighter than one against the fp32 oracle, which differs from the kernels by BF16 rounding at every layer.

Rounding points, as read from the kernel source:
  * weights: BF16 by round-to-nearest-even, f2bf (srfbn.cu pack_*: f2bf); biases stay fp32;
  * every igemm_kernel layer output (conv_in, the 1x1 layers, both transposed convs, the x2 strided conv, the x4
    downtran): x_b = bf16(acc + bias), then PReLU in packed BF16 with the slope rounded to BF16 (igemm.cuh
    make_prelu / prelu_pack / convert32 / convert16): slope in [0,1]: max(x_b, bf16(x_b*s_b)); slope > 1:
    min(x_b, bf16(x_b*s_b)); slope < 0: bf16(s_b*min(x_b,0) + max(x_b,0)) (hfma2, one rounding).  The form is picked
    on the fp32 slope;
  * conv_in's input: bf16(x + sub_bias), and the 3x3 zero padding is a zero of the SHIFTED image (srfbn.cu
    im2col_kernel);
  * x4 feedback groups: U (the transposed conv) and every hr[i] are BF16 -- also where fused_updown_kernel keeps U on
    chip (fused_down.cuh, MERGED branch: convert32 of T_U); the downtran output H is rounded to BF16 on chip
    (fused_down.cuh: convert32 into s_h); the 8x8-s4 conv sums in fp32 across its partial slots and
    finalize_lr_kernel, and lr[i+1] = bf16(PReLU(acc + bias)) with the PReLU in fp32 and the fp32 slope, NOT the
    packed form (fused_down.cuh: `prelu(comb[0][k] + below[k] + s_down[..], slope, 1)` and finalize_lr_kernel's
    `prelu(r[k] + bias, slope, 1)`, then pack_bf16);
  * x2 feedback groups: deconv2, the downtran over HR rows and downconv2 each output BF16 with the packed PReLU
    (EPI_DECONV2 convert32, EPI_ROWS convert32, EPI_DOWN2 convert16);
  * conv_out (EPI_CONV_OUT): BF16 input (the `out` map) and weights, fp32 output = skip + (bias + 9 tap partials) +
    add_mean, with the bilinear skip taken from the UNROUNDED fp32 x + sub_bias;
  * fc fuse: fp32 throughout (fc_fuse_kernel), restated here in float64.

torch converts float64 to bfloat16 through float; round_bf16 does the same explicitly (fp64 -> fp32 -> f2bf).  The
double rounding this causes is negligible next to the fp32-versus-fp64 difference of the accumulations.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle.srfbn_oracle import GEOMETRY


def f2bf_bits(t: torch.Tensor) -> torch.Tensor:
    """srfbn.cu f2bf on the fp32 value of t: the BF16 bit pattern (int64, 0..0xffff), round to nearest even; NaN keeps
    its sign and top payload bits and gets the quiet bit (u >> 16 | 0x40)."""
    u = t.to(torch.float32).contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    nan = (u & 0x7FFFFFFF) > 0x7F800000
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) & 0xFFFF
    return torch.where(nan, ((u >> 16) | 0x40) & 0xFFFF, r)


def bits_to_float(bits: torch.Tensor) -> torch.Tensor:
    """BF16 bit patterns (any integer dtype, 0..0xffff) -> their values as float64."""
    b = bits.to(torch.int64) & 0xFFFF
    return (((b ^ 0x8000) - 0x8000) << 16).to(torch.int32).view(torch.float32).to(torch.float64)


def round_bf16(t: torch.Tensor) -> torch.Tensor:
    """t rounded to BF16 as the kernels and the weight packing round (fp32, then f2bf), returned as float64."""
    return bits_to_float(f2bf_bits(t))


class Restatement:
    """Options of one restatement.  rounding=False drops every BF16 rounding (the float64 oracle); the other switches
    each re-introduce one specific error, so a test can show that its bound rejects it:
      pad_unshifted: conv_in pads x with zeros before sub_mean (the padding is then sub_bias, not 0);
      skip_zero_ext: the bilinear skip reads zeros outside the LR image instead of clamping to its border;
      exact_slopes:  state-dict prefixes whose packed-BF16 PReLU uses the fp32 slope instead of the rounded one."""

    def __init__(self, rounding=True, pad_unshifted=False, skip_zero_ext=False, exact_slopes=()):
        self.rounding = rounding
        self.pad_unshifted = pad_unshifted
        self.skip_zero_ext = skip_zero_ext
        self.exact_slopes = set(exact_slopes)

    def rb(self, t):
        return round_bf16(t) if self.rounding else t

    def weight(self, sd, prefix, dev):
        return self.rb(sd[prefix + ".0.weight"].to(dev, torch.float64))

    def bias(self, sd, prefix, dev):
        return sd[prefix + ".0.bias"].to(dev, torch.float64)

    def slope(self, sd, prefix):
        return float(sd[prefix + ".1.weight"].reshape(-1)[0].to(torch.float32))

    def act_packed(self, v, sd, prefix):
        """bf16(acc + bias) -> packed-BF16 PReLU (igemm.cuh prelu_pack)."""
        s = self.slope(sd, prefix)
        if not self.rounding:
            return torch.where(v >= 0, v, v * s)
        sb = s if prefix in self.exact_slopes else float(round_bf16(torch.tensor(s)))
        return prelu_packed(self.rb(v), s, sb)

    def act_fp32(self, v, sd, prefix):
        """bf16(PReLU(acc + bias)) with the fp32 slope (fused_down.cuh / finalize_lr_kernel)."""
        s = self.slope(sd, prefix)
        return self.rb(torch.where(v >= 0, v, v * s))

    # -- layers ---------------------------------------------------------------------------------------------------
    def conv_in(self, x, sd):
        """x (B,3,h,w) 0..255 -> (B,128,h,w): sub_mean, 3x3 p1 over the shifted image, PReLU."""
        dev = x.device
        sb = sd["sub_mean.bias"].to(dev, torch.float64).view(1, 3, 1, 1)
        if self.pad_unshifted:
            xs = self.rb(F.pad(x, (1, 1, 1, 1)) + sb)
            pad = 0
        else:
            xs = self.rb(x + sb)
            pad = 1
        v = F.conv2d(xs, self.weight(sd, "conv_in", dev), self.bias(sd, "conv_in", dev), padding=pad)
        return self.act_packed(v, sd, "conv_in")

    def pointwise(self, x, sd, prefix):
        dev = x.device
        return self.act_packed(F.conv2d(x, self.weight(sd, prefix, dev), self.bias(sd, prefix, dev)), sd, prefix)

    def up(self, x, sd, prefix, scale):
        _, st, pd = GEOMETRY[scale]
        dev = x.device
        v = F.conv_transpose2d(x, self.weight(sd, prefix, dev), self.bias(sd, prefix, dev), stride=st, padding=pd)
        return self.act_packed(v, sd, prefix)

    def down(self, x, sd, prefix, scale):
        _, st, pd = GEOMETRY[scale]
        dev = x.device
        v = F.conv2d(x, self.weight(sd, prefix, dev), self.bias(sd, prefix, dev), stride=st, padding=pd)
        return self.act_packed(v, sd, prefix) if scale == 2 else self.act_fp32(v, sd, prefix)

    def skip(self, x, sd, scale):
        """Bilinear (align_corners=False) upsampling of the unrounded x + sub_bias (igemm.cuh EPI_CONV_OUT)."""
        dev = x.device
        xs = x + sd["sub_mean.bias"].to(dev, torch.float64).view(1, 3, 1, 1)
        if not self.skip_zero_ext:
            return F.interpolate(xs, scale_factor=scale, mode="bilinear", align_corners=False)
        h, w = xs.shape[-2:]
        xp = F.pad(xs, (1, 1, 1, 1))                  # zero ring: index i of the image is i + 1 here

        def taps(n):
            src = (torch.arange(scale * n, dtype=torch.float64, device=dev) + 0.5) / scale - 0.5
            i0 = torch.floor(src)
            return i0.long() + 1, i0.long() + 2, src - i0

        y0, y1, ly = taps(h)
        x0, x1, lx = taps(w)
        ly, lx = ly.view(-1, 1), lx.view(1, -1)
        r0, r1 = xp[:, :, y0], xp[:, :, y1]
        return ((1 - ly) * ((1 - lx) * r0[..., x0] + lx * r0[..., x1])
                + ly * ((1 - lx) * r1[..., x0] + lx * r1[..., x1]))

    def conv_out(self, hb, x, sd, scale):
        """hb (B,32,sH,sW) BF16 values, x (B,3,h,w) -> (B,3,sH,sW) fp32-path output: conv + skip + add_mean."""
        dev = hb.device
        y = F.conv2d(hb, self.rb(sd["conv_out.0.weight"].to(dev, torch.float64)),
                     sd["conv_out.0.bias"].to(dev, torch.float64), padding=1)
        return self.skip(x, sd, scale) + y + sd["add_mean.bias"].to(dev, torch.float64).view(1, 3, 1, 1)

    def feedback_block(self, x, last_hidden, sd, num_groups, scale):
        """srfbn_oracle.feedback_block with the kernels' rounding points."""
        x = self.pointwise(torch.cat((x, last_hidden), 1), sd, "block.compress_in")
        lr, hr = [x], []
        for i in range(num_groups):
            ld_l = torch.cat(lr[: i + 1], 1)
            if i > 0:
                ld_l = self.pointwise(ld_l, sd, f"block.uptranBlocks.{i - 1}")
            hr.append(self.up(ld_l, sd, f"block.upBlocks.{i}", scale))
            ld_h = torch.cat(hr[: i + 1], 1)
            if i > 0:
                ld_h = self.pointwise(ld_h, sd, f"block.downtranBlocks.{i - 1}")
            lr.append(self.down(ld_h, sd, f"block.downBlocks.{i}", scale))
        return self.pointwise(torch.cat(lr[1:], 1), sd, "block.compress_out")

    def forward_maps(self, x, sd, num_steps=3, num_groups=6, upscale=4):
        """x (M,3,h,w) 0..255 (any float dtype; computed in float64 on x.device) -> per-map images (M,3,sH,sW)."""
        x = x.to(torch.float64)
        with torch.no_grad():
            f = self.pointwise(self.conv_in(x, sd), sd, "feat_in")
            hidden = f
            for _ in range(num_steps):
                hidden = self.feedback_block(f, hidden, sd, num_groups, upscale)
            return self.conv_out(self.up(hidden, sd, "out", upscale), x, sd, upscale)


def prelu_packed(xb, slope, sb):
    """The packed-BF16 PReLU of igemm.cuh prelu_pack on BF16 values xb (float64): the form is picked on the fp32
    `slope`, the arithmetic uses its BF16 rounding `sb`."""
    if 0.0 <= slope <= 1.0:
        return torch.maximum(xb, round_bf16(xb * sb))
    if slope > 1.0:
        return torch.minimum(xb, round_bf16(xb * sb))
    return round_bf16(sb * torch.clamp(xb, max=0.0) + torch.clamp(xb, min=0.0))


def forward_maps(x, sd, num_steps=3, num_groups=6, upscale=4, **options):
    """Per-map images (M,3,sH,sW) float64 of the BF16-faithful restatement; options: see Restatement."""
    return Restatement(**options).forward_maps(x, sd, num_steps, num_groups, upscale)


def fc_fuse(maps, sd):
    """srfbn_oracle.fc_fuse in float64: maps (M,3,H,W) -> (1,3,H,W)."""
    dev = maps.device
    t = maps.to(torch.float64).permute(1, 2, 3, 0)
    t = F.relu(F.linear(t, sd["fc.0.weight"].to(dev, torch.float64), sd["fc.0.bias"].to(dev, torch.float64)))
    t = F.relu(F.linear(t, sd["fc.2.weight"].to(dev, torch.float64), sd["fc.2.bias"].to(dev, torch.float64)))
    return t.permute(3, 0, 1, 2)
