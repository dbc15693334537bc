"""The CPU restatement of the correlation kernels (oracle.or_correlation with padded=1, or_correlation_backward_chain):
the arithmetic that test_correlation_faithful_gpu holds correlation.cu to bit for bit.  No GPU.

An independent numpy restatement (the correctly rounded `_fmaf` of test_front_fast_restatement) must give the C
restatement's bits; the same numpy code with the FMAs split into a product and a sum, with the channels taken outside the
window taps, or with the backward's displacement loops swapped, must not.  The padded rule (the reference's zero-padded
copies, every product taken) turns 0 * Inf into NaN where the skipping rule does not, and both stay within a bound
derived from the arithmetic of an fp64 evaluation."""
import numpy as np
import pytest

from oracle import oracle as orc
from tests.test_front_fast_restatement import _fmaf

F32, F64 = np.float32, np.float64
U = 2.0 ** -24                  # unit roundoff of fp32


def _geometry(H, W, pad, k, md, s1, s2):
    border = (k - 1) // 2 + md
    outH = -(-(H + 2 * pad - 2 * border) // s1)
    outW = -(-(W + 2 * pad - 2 * border) // s1)
    R = md // s2
    return outH, outW, R, 2 * R + 1


def _at(img, yy, xx):
    """img (B,C,H,W) at rows yy (n,) and columns xx (m,): (B,C,n,m) with zeros outside the image, and the mask."""
    H, W = img.shape[2:]
    ok = ((yy >= 0) & (yy < H))[:, None] & ((xx >= 0) & (xx < W))[None, :]
    v = img[:, :, np.clip(yy, 0, H - 1)][:, :, :, np.clip(xx, 0, W - 1)]
    return np.where(ok, v, 0).astype(img.dtype), ok


def _fma_for(variant):
    if variant == "unfused":
        return lambda x, y, z: ((x * y).astype(F32) + z).astype(F32)
    return _fmaf


def _corr_np(a, b, pad, k, md, s1, s2, padded=True, variant="faithful"):
    """numpy restatement of the forward.  variant: "faithful" (one fmaf chain over (j, i) then c), "unfused" (each fmaf
    a rounded product and a rounded sum), "c_outer" (the channels outside the window taps)."""
    B, C, H, W = a.shape
    outH, outW, R, D = _geometry(H, W, pad, k, md, s1, s2)
    krad = (k - 1) // 2
    ys, xs = np.arange(outH) * s1 + md - pad, np.arange(outW) * s1 + md - pad
    fma = _fma_for(variant)
    out = np.empty((B, D * D, outH, outW), F32)
    taps = [(j, i) for j in range(-krad, krad + 1) for i in range(-krad, krad + 1)]
    steps = [(t, c) for t in range(len(taps)) for c in range(C)]
    if variant == "c_outer":
        steps = [(t, c) for c in range(C) for t in range(len(taps))]
    for tj in range(-R, R + 1):
        for ti in range(-R, R + 1):
            v = []
            for j, i in taps:
                v1, ok1 = _at(a, ys + j, xs + i)
                v2, ok2 = _at(b, ys + j + tj * s2, xs + i + ti * s2)
                v.append((v1, v2, ok1 & ok2))
            acc = np.zeros((B, outH, outW), F32)
            for t, c in steps:
                v1, v2, ok = v[t]
                nxt = fma(v1[:, c], v2[:, c], acc)
                acc = nxt if padded else np.where(ok, nxt, acc).astype(F32)
            out[:, (tj + R) * D + ti + R] = acc / F32(k * k * C)
    return out


def _corr_bwd_np(a, b, g, pad, k, md, s2, which, variant="faithful"):
    """numpy restatement of correlation_backward_kernel for gradInput1 (which=0) / gradInput2 (which=1).  variant:
    "faithful" (tj, then ti, then the window rows and columns), "unfused", "ti_outer" (ti before tj)."""
    B, C, H, W = a.shape
    outH, outW = g.shape[2:]
    R, D, krad = md // s2, 2 * (md // s2) + 1, (k - 1) // 2
    other = b if which == 0 else a
    y, x = np.arange(H) + pad, np.arange(W) + pad
    fma = _fma_for(variant)
    order = [(tj, ti) for tj in range(D) for ti in range(D)]
    if variant == "ti_outer":
        order = [(tj, ti) for ti in range(D) for tj in range(D)]
    acc = np.zeros(a.shape, F32)
    for tj, ti in order:
        j2, i2 = (tj - R) * s2, (ti - R) * s2
        val, _ = _at(other, (y - j2 if which else y + j2) - pad, (x - i2 if which else x + i2) - pad)
        ymin = y - krad - md - (j2 if which else 0)
        xmin = x - krad - md - (i2 if which else 0)
        for dj in range(2 * krad + 1):
            for di in range(2 * krad + 1):
                gv, ok = _at(g[:, None, tj * D + ti], ymin + dj, xmin + di)       # (B,1,H,W): one window output
                acc = np.where(ok, fma(gv, val, acc), acc).astype(F32)
    return acc / F32(k * k * C)


def _bits(x):
    """int32 view with every NaN mapped to one value: x86 and CUDA NaN payloads differ."""
    x = np.asarray(x, F32)
    return np.where(np.isnan(x), np.int32(0x7FC00000), x.view(np.int32))


def _case(seed, shape, scale=1.0):
    rng = np.random.default_rng(seed)
    return tuple((rng.standard_normal(shape) * scale).astype(F32) for _ in range(2))


# (B, C, H, W, pad, k, md, s1, s2): k = 1 and 3, s1 = 1 and 2, s2 = 1 and 2, pad <, = and > max_displacement
FWD = [
    (2, 5, 9, 13, 4, 1, 4, 1, 2),       # pad = md, the FlowNetC rule
    (1, 3, 11, 12, 2, 1, 4, 1, 2),      # pad < md: the output shrinks
    (1, 4, 8, 9, 6, 1, 3, 1, 1),        # pad > md: whole padded rows and columns in the output
    (1, 3, 10, 11, 3, 3, 2, 1, 1),      # 3x3 window, pad = md + krad
    (1, 2, 9, 10, 1, 3, 2, 1, 2),       # 3x3 window, pad < md
    (2, 3, 11, 13, 5, 3, 3, 2, 1),      # 3x3 window, strided outputs, pad > md + krad
    (1, 4, 12, 9, 2, 1, 3, 2, 2),       # strided outputs, md not a multiple of s2
]


@pytest.mark.parametrize("cfg", FWD)
@pytest.mark.parametrize("padded", [True, False])
def test_forward_numpy_restatement_matches_c_bit_for_bit(cfg, padded):
    B, C, H, W, pad, k, md, s1, s2 = cfg
    a, b = _case(sum(cfg), (B, C, H, W))
    want = _corr_np(a, b, pad, k, md, s1, s2, padded)
    got = orc.correlation(a, b, pad, k, md, s1, s2, padded=padded)
    assert np.array_equal(got.view(np.int32), want.view(np.int32))
    assert np.abs(got).max() > 0
    # row fan-out and item range restate the same bits
    assert np.array_equal(orc.correlation(a, b, pad, k, md, s1, s2, padded=padded, threads=3).view(np.int32),
                          got.view(np.int32))
    assert np.array_equal(orc.correlation(a, b, pad, k, md, s1, s2, padded=padded, items=(B - 1, B)).view(np.int32),
                          got[B - 1:].view(np.int32))


@pytest.mark.parametrize("cfg", [c for c in FWD if c[7] == 1])
def test_backward_numpy_restatement_matches_c_bit_for_bit(cfg):
    B, C, H, W, pad, k, md, _, s2 = cfg
    a, b = _case(sum(cfg) + 1, (B, C, H, W))
    outH, outW, _, D = _geometry(H, W, pad, k, md, 1, s2)
    g = np.random.default_rng(sum(cfg) + 2).standard_normal((B, D * D, outH, outW)).astype(F32)
    g1, g2 = orc.correlation_backward_chain(a, b, g, pad, k, md, s2)
    for which, got in ((0, g1), (1, g2)):
        want = _corr_bwd_np(a, b, g, pad, k, md, s2, which)
        assert np.array_equal(got.view(np.int32), want.view(np.int32)), which
        assert np.abs(got).max() > 0
    c0 = C // 2
    p1, p2 = orc.correlation_backward_chain(a, b, g, pad, k, md, s2, items=(B - 1, B), channels=(c0, C), threads=2)
    assert np.array_equal(p1.view(np.int32), g1[B - 1:, c0:].view(np.int32))
    assert np.array_equal(p2.view(np.int32), g2[B - 1:, c0:].view(np.int32))


def test_unfused_and_reordered_restatements_give_other_bits():
    """The comparison is sharp enough to tell the kernels' arithmetic from its neighbours."""
    a, b = _case(11, (1, 8, 10, 11))
    want = orc.correlation(a, b, 3, 3, 2, 1, 1, padded=True)
    for variant in ("unfused", "c_outer"):
        other = _corr_np(a, b, 3, 3, 2, 1, 1, True, variant)
        assert not np.array_equal(other.view(np.int32), want.view(np.int32)), variant
        assert np.abs(other - want).max() <= 1e-5                     # same value to fp32 rounding
    a, b = _case(12, (1, 8, 9, 12))
    outH, outW, _, D = _geometry(9, 12, 4, 1, 4, 1, 2)
    g = np.random.default_rng(13).standard_normal((1, D * D, outH, outW)).astype(F32)
    g1, g2 = orc.correlation_backward_chain(a, b, g, 4, 1, 4, 2)
    for which, want in ((0, g1), (1, g2)):
        for variant in ("unfused", "ti_outer"):
            other = _corr_bwd_np(a, b, g, 4, 1, 4, 2, which, variant)
            assert not np.array_equal(other.view(np.int32), want.view(np.int32)), (which, variant)


def test_padded_rule_turns_zero_times_inf_into_nan():
    """An Inf of in2 that only meets in1's padding (and vice versa) is NaN under the reference's zero padding and
    invisible under the skipping rule; an Inf that meets a real value is +-Inf under both."""
    B, C, H, W, pad, k, md, s1, s2 = 1, 3, 8, 9, 6, 1, 4, 1, 2
    outH, outW, R, D = _geometry(H, W, pad, k, md, s1, s2)
    a, b = _case(21, (B, C, H, W))
    b[0, 1, 0, 0] = np.inf                # in2 (0, 0): in1 is padding wherever output row y - 2 < 0 meets it
    a[0, 2, H - 1, W - 1] = -np.inf       # in1 (H-1, W-1): in2 is padding for displacements past the corner
    with np.errstate(invalid="ignore", over="ignore"):
        pad_out = orc.correlation(a, b, pad, k, md, s1, s2, padded=True)
        skip = orc.correlation(a, b, pad, k, md, s1, s2, padded=False)
        assert np.array_equal(_bits(pad_out), _bits(_corr_np(a, b, pad, k, md, s1, s2, True)))
        assert np.array_equal(_bits(skip), _bits(_corr_np(a, b, pad, k, md, s1, s2, False)))
    # output (y, x) = in1 (y - 2, x - 2); displacement (tj, ti) reads in2 at (y - 2 + 2 tj, x - 2 + 2 ti)
    # in2 (0, 0) from in1 (-2, -2) (padding) at tj = ti = 1: output (0, 0), channel (1 + R) * D + 1 + R
    ch = (1 + R) * D + 1 + R
    assert np.isnan(pad_out[0, ch, 0, 0]) and np.isfinite(skip[0, ch, 0, 0])
    # in1 (H-1, W-1) = output (H+1, W+1) against in2 (H+1, W+1) (padding) at tj = ti = 1
    assert np.isnan(pad_out[0, ch, H + 1, W + 1]) and np.isfinite(skip[0, ch, H + 1, W + 1])
    # real meets real: the same non-finite value under both rules
    assert np.isinf(pad_out[0, R * D + R, 2, 2]) and np.isinf(skip[0, R * D + R, 2, 2])
    assert np.array_equal(np.isnan(skip), np.zeros_like(skip, bool))
    finite = np.isfinite(pad_out) & np.isfinite(skip)
    assert np.array_equal(pad_out[finite].view(np.int32), skip[finite].view(np.int32))


def test_backward_grad_inf_meeting_padding_is_nan():
    """An Inf of grad_output at an output whose displacement reads the other image's padding: the element of the
    gradient that sums that output is NaN (0 * Inf), in the kernel order and in the reference order."""
    B, C, H, W, pad, k, md, s2 = 1, 2, 7, 8, 4, 1, 4, 2
    outH, outW, R, D = _geometry(H, W, pad, k, md, 1, s2)
    a, b = _case(31, (B, C, H, W))
    g = np.random.default_rng(32).standard_normal((B, D * D, outH, outW)).astype(F32)
    # output (0, 0) is in1 (0, 0) (pad = md); displacement (tj, ti) = (0, 0) reads in2 (-2R, -2R): padding
    g[0, 0, 0, 0] = np.inf
    with np.errstate(invalid="ignore", over="ignore"):
        g1, g2 = orc.correlation_backward_chain(a, b, g, pad, k, md, s2)
        r1, r2 = orc.correlation_backward(a, b, g, pad, k, md, s2)
        want1 = _corr_bwd_np(a, b, g, pad, k, md, s2, 0)
    assert np.isnan(g1[0, :, 0, 0]).all() and np.isnan(r1[0, :, 0, 0]).all()
    assert np.isfinite(np.delete(g1.reshape(C, -1), 0, axis=1)).all()
    assert np.isfinite(g2).all()            # gradInput2's pixel of that product is outside in2
    assert np.array_equal(_bits(g1), _bits(want1))


def _gamma(n):
    return n * U / (1 - n * U)


@pytest.mark.parametrize("cfg", FWD[:4])
def test_restatement_within_derived_bound_of_fp64(cfg):
    """|fp32 restatement - fp64| <= gamma_{n+1} * sum|products| / N per output: n fmaf roundings of a chain of n
    products (n = N = k*k*C for the forward; the number of window products for the backward) and one division."""
    B, C, H, W, pad, k, md, s1, s2 = cfg
    a, b = _case(sum(cfg) + 40, (B, C, H, W), scale=3.0)
    N = k * k * C
    got = orc.correlation(a, b, pad, k, md, s1, s2, padded=True).astype(F64)
    a64, b64 = a.astype(F64), b.astype(F64)
    exact = _corr_np_f64(a64, b64, pad, k, md, s1, s2)
    mag = _corr_np_f64(np.abs(a64), np.abs(b64), pad, k, md, s1, s2)
    assert (np.abs(got - exact) <= _gamma(N + 1) * mag).all()
    assert (np.abs(got - exact) > 0).any()
    if s1 == 1:
        outH, outW, _, D = _geometry(H, W, pad, k, md, 1, s2)
        g = (np.random.default_rng(sum(cfg) + 41).standard_normal((B, D * D, outH, outW)) * 2).astype(F32)
        chain = orc.correlation_backward_chain(a, b, g, pad, k, md, s2)
        ref_order = orc.correlation_backward(a, b, g, pad, k, md, s2)
        n = D * D * k * k
        for which in (0, 1):
            ex = _corr_bwd_np_f64(a64, b64, g.astype(F64), pad, k, md, s2, which)
            mg = _corr_bwd_np_f64(np.abs(a64), np.abs(b64), np.abs(g.astype(F64)), pad, k, md, s2, which)
            for r in (chain[which], ref_order[which]):
                assert (np.abs(r.astype(F64) - ex) <= _gamma(n + 1) * mg).all(), which


def _corr_np_f64(a, b, pad, k, md, s1, s2):
    B, C, H, W = a.shape
    outH, outW, R, D = _geometry(H, W, pad, k, md, s1, s2)
    krad = (k - 1) // 2
    ys, xs = np.arange(outH) * s1 + md - pad, np.arange(outW) * s1 + md - pad
    out = np.zeros((B, D * D, outH, outW), F64)
    for tj in range(-R, R + 1):
        for ti in range(-R, R + 1):
            for j in range(-krad, krad + 1):
                for i in range(-krad, krad + 1):
                    v1, _ = _at(a, ys + j, xs + i)
                    v2, _ = _at(b, ys + j + tj * s2, xs + i + ti * s2)
                    out[:, (tj + R) * D + ti + R] += (v1 * v2).sum(1)
    return out / (k * k * C)


def _corr_bwd_np_f64(a, b, g, pad, k, md, s2, which):
    B, C, H, W = a.shape
    R, D, krad = md // s2, 2 * (md // s2) + 1, (k - 1) // 2
    other = b if which == 0 else a
    y, x = np.arange(H) + pad, np.arange(W) + pad
    acc = np.zeros(a.shape, F64)
    for tj in range(D):
        for ti in range(D):
            j2, i2 = (tj - R) * s2, (ti - R) * s2
            val, _ = _at(other, (y - j2 if which else y + j2) - pad, (x - i2 if which else x + i2) - pad)
            for dj in range(2 * krad + 1):
                for di in range(2 * krad + 1):
                    gv, _ = _at(g[:, None, tj * D + ti], y - krad - md - (j2 if which else 0) + dj,
                                x - krad - md - (i2 if which else 0) + di)
                    acc += gv * val
    return acc / (k * k * C)
