"""GPU: the REFERENCE's own CUDA ops (compiled from /root/reference into oracle/_ref by
oracle/build_ref.py) against the C oracle and against the product kernels, bit for bit.
This is the pin of oracle.c::or_resample2d / or_channelnorm (the reference has no tests).
Without the compiled ops, the same comparisons run against their stored outputs (tests/ref_pins.py)."""
import numpy as np
import pytest
import torch

from oracle import build_ref
from oracle import oracle as orc
from tests import ref_pins as pin
from video_super_resolution_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _ref(name):
    """The reference's compiled op, or None: then the tests compare with its pinned outputs."""
    return build_ref.load_ref(name)


@pytest.mark.parametrize("shape", [(1, 3, 64, 64), (2, 3, 256, 448), (1, 2, 33, 47)])
@pytest.mark.parametrize("bilinear", [True, False])
def test_reference_resample2d_equals_oracle_and_product(shape, bilinear, request):
    ref = _ref("resample2d_cuda")
    B, C, H, W = shape
    g = torch.Generator().manual_seed(H)
    img = (torch.rand(shape, generator=g) * 255).to(DEV)
    flow = ((torch.rand((B, 2, H, W), generator=g) - 0.5) * 30).to(DEV)
    want = None
    if ref is not None:
        out = torch.zeros_like(img)                      # resample2d.py:19
        ref.forward(img, flow, out, 1, bilinear)         # resample2d.py:21
        torch.cuda.synchronize()
        want = out.cpu().numpy()
    pin.assert_equal(request.node.name, orc.resample2d_nchw(img.cpu().numpy(), flow.cpu().numpy(), 1, bilinear), want)
    pin.assert_equal(request.node.name, ops.resample2d(img, flow, 1, bilinear), want)


@pytest.mark.parametrize("shape", [(1, 3, 64, 64), (2, 2, 100, 37)])
def test_reference_channelnorm_equals_oracle_and_product(shape, request):
    ref = _ref("channelnorm_cuda")
    x = (torch.randn(shape, generator=torch.Generator().manual_seed(1)) * 20).to(DEV)
    want = None
    if ref is not None:
        out = torch.zeros((shape[0], 1, shape[2], shape[3]), device=DEV)
        ref.forward(x, out, 2)                           # channelnorm.py:14
        torch.cuda.synchronize()
        want = out.cpu().numpy()
    pin.assert_equal(request.node.name, orc.channelnorm_nchw(x.cpu().numpy()), want)
    pin.assert_equal(request.node.name, ops.channelnorm(x), want)


def test_golden_gpu_fixture_if_present(golden_dir):
    """Fixtures produced by tests/golden/make_golden_gpu.py from the reference ops on a B200."""
    import os
    path = os.path.join(golden_dir, "resample2d_ref.npz")
    if not os.path.exists(path):
        pytest.skip("resample2d_ref.npz not generated yet")
    z = np.load(path)
    for mode, bil in (("bilinear", True), ("nearest", False)):
        got = ops.resample2d(torch.from_numpy(z["img"]).to(DEV), torch.from_numpy(z["flow"]).to(DEV), 1, bil)
        assert np.array_equal(got.cpu().numpy(), z[mode])
    got = ops.channelnorm(torch.from_numpy(z["img"]).to(DEV))
    assert np.array_equal(got.cpu().numpy(), z["channelnorm"])


@pytest.mark.parametrize("shape", [(1, 3, 64, 64), (2, 2, 33, 47), (1, 5, 40, 120)])
def test_reference_resample2d_backward_equals_oracle_and_product(shape, request):
    """resample2d_cuda.backward of the reference binary (resample2d_kernel.cu:75-198) vs oracle vs product.
    grad_input2 is deterministic -> bit for bit; grad_input1 is an atomic scatter -> fp32 order tolerance."""
    ref = _ref("resample2d_cuda")
    B, C, H, W = shape
    g = torch.Generator().manual_seed(H + C)
    img = (torch.rand(shape, generator=g) * 255).to(DEV)
    flow = ((torch.rand((B, 2, H, W), generator=g) - 0.5) * 30).to(DEV)      # negative coords: int() != floor
    gout = torch.randn(shape, generator=g).to(DEV)
    r1 = r2 = None
    if ref is not None:
        r1, r2 = torch.zeros_like(img), torch.zeros_like(flow)                   # resample2d.py:32-33
        ref.backward(img, flow, gout, r1, r2, 1, True)                           # resample2d.py:35-37
        torch.cuda.synchronize()
    o1, o2 = orc.resample2d_backward(img.cpu().numpy(), flow.cpu().numpy(), gout.cpu().numpy())
    p1, p2 = ops.resample2d_backward(img, flow, gout)
    name = request.node.name
    pin.assert_equal(name + "/grad_input2", o2, r2)
    pin.assert_equal(name + "/grad_input2", p2, r2)
    tol = pin.assert_close(name + "/grad_input1", o1, r1)
    pin.assert_close(name + "/grad_input1", p1, r1)
    assert np.abs(p1.cpu().numpy() - o1).max() <= 2 * tol


@pytest.mark.parametrize("shape", [(1, 3, 64, 64), (2, 2, 100, 37)])
def test_reference_channelnorm_backward_equals_oracle_and_product(shape, request):
    ref = _ref("channelnorm_cuda")
    g = torch.Generator().manual_seed(2)
    x = (torch.randn(shape, generator=g) * 20).to(DEV)
    x[0, :, 0, 0] = 0.0                                                      # zero norm: the +1e-9 guard
    out = ops.channelnorm(x)
    gout = torch.randn(out.shape, generator=g).to(DEV)
    want = None
    if ref is not None:
        r = torch.zeros_like(x)
        ref.backward(x, out, gout, r, 2)                                         # channelnorm.py:25-26
        torch.cuda.synchronize()
        want = r.cpu().numpy()
    pin.assert_equal(request.node.name, orc.channelnorm_backward(x.cpu().numpy(), out.cpu().numpy(), gout.cpu().numpy()), want)
    pin.assert_equal(request.node.name, ops.channelnorm_backward(x, out, gout), want)


def test_autograd_function_surfaces_backward():
    """Resample2d / ChannelNorm modules differentiate like the reference's Functions (resample2d.py:25-39)."""
    from video_super_resolution_b200.my_packages.FlowProjection.networks.channelnorm_package.channelnorm import ChannelNorm
    from video_super_resolution_b200.my_packages.FlowProjection.networks.resample2d_package.resample2d import Resample2d
    g = torch.Generator().manual_seed(3)
    img = (torch.rand((1, 3, 24, 32), generator=g) * 255).to(DEV).requires_grad_(True)
    flow = ((torch.rand((1, 2, 24, 32), generator=g) - 0.5) * 6).to(DEV).requires_grad_(True)
    y = ChannelNorm()(Resample2d()(img, flow))
    y.sum().backward()
    assert img.grad is not None and flow.grad is not None
    assert torch.isfinite(img.grad).all() and torch.isfinite(flow.grad).all()
    # a finite-difference check of the flow gradient away from integer crossings
    with torch.no_grad():
        eps = 1e-2
        f2 = flow.detach().clone()
        f2[0, 0, 10, 10] += eps
        num = (ChannelNorm()(Resample2d()(img.detach(), f2)).sum() - y.detach().sum()) / eps
    assert abs(num.item() - flow.grad[0, 0, 10, 10].item()) <= 0.05 * abs(num.item()) + 0.5


@pytest.mark.parametrize("cfg", [
    dict(shape=(1, 64, 24, 40), pad=20, k=1, md=20, s1=1, s2=2),      # FlowNetC (FlowNetC.py:22), fewer channels
    dict(shape=(2, 256, 16, 24), pad=20, k=1, md=20, s1=1, s2=2),     # FlowNetC channels
    dict(shape=(1, 16, 20, 28), pad=5, k=3, md=4, s1=1, s2=1),        # 3x3 kernel window (pad >= md + 1: with a
                                                                      # smaller pad the reference reads outside its padded copy)
    dict(shape=(1, 8, 21, 37), pad=4, k=1, md=4, s1=2, s2=2),         # strided outputs
    dict(shape=(1, 20, 9, 300), pad=20, k=1, md=20, s1=1, s2=2),      # register-tiled path: 3 x-tiles, ragged, C % 8 != 0
    dict(shape=(2, 12, 11, 70), pad=8, k=1, md=8, s1=1, s2=2),        # register-tiled path with D = 9
])
def test_reference_correlation_equals_oracle_and_product(cfg, request):
    """correlation_cuda.forward of the reference binary (correlation_cuda_kernel.cu:46-147) vs oracle vs product;
    fp32 summation order differs (32 strided partials + shuffle tree there), so compare to 1e-5 relative."""
    ref = _ref("correlation_cuda")
    g = torch.Generator().manual_seed(cfg["shape"][1])
    a = torch.randn(cfg["shape"], generator=g).to(DEV)
    b = torch.randn(cfg["shape"], generator=g).to(DEV)
    want = None
    if ref is not None:
        r1, r2, out = a.new_empty(0), a.new_empty(0), a.new_empty(0)                # correlation.py:22-24
        ref.forward(a, b, r1, r2, out, cfg["pad"], cfg["k"], cfg["md"], cfg["s1"], cfg["s2"], 1)
        torch.cuda.synchronize()
        want = out.cpu().numpy()
    got = ops.correlation(a, b, cfg["pad"], cfg["k"], cfg["md"], cfg["s1"], cfg["s2"], 1).cpu().numpy()
    orc_out = orc.correlation(a.cpu().numpy(), b.cpu().numpy(), cfg["pad"], cfg["k"], cfg["md"], cfg["s1"], cfg["s2"])
    tol = pin.assert_close(request.node.name, orc_out, want)
    pin.assert_close(request.node.name, got, want)
    assert got.shape == orc_out.shape and np.abs(got - orc_out).max() <= 2 * tol


def test_correlation_register_tiled_path_is_bit_identical_to_generic_kernel(monkeypatch):
    """kernel_size 1 / stride1 1 / stride2 2 (FlowNetC.py:22) takes the register-tiled kernel; it keeps the generic
    kernel's fp32 FMA chain in channel order, so the two agree bit for bit (also with pad < max_displacement, where
    the output shrinks and the window centres start inside the image)."""
    g = torch.Generator().manual_seed(7)
    for shape, pad, md in (((1, 37, 30, 150), 20, 20), ((2, 16, 50, 90), 6, 10)):
        a = torch.randn(shape, generator=g).to(DEV)
        b = torch.randn(shape, generator=g).to(DEV)
        monkeypatch.delenv("VSR_CORR_GENERIC", raising=False)
        fast = ops.correlation(a, b, pad, 1, md, 1, 2, 1)
        monkeypatch.setenv("VSR_CORR_GENERIC", "1")
        slow = ops.correlation(a, b, pad, 1, md, 1, 2, 1)
        assert torch.equal(fast, slow)
        assert fast.abs().max().item() > 0


@pytest.mark.parametrize("cfg", [
    dict(shape=(1, 8, 24, 40), pad=20, k=1, md=20, s2=2),          # FlowNetC geometry (FlowNetC.py:22)
    dict(shape=(2, 5, 13, 21), pad=8, k=1, md=8, s2=2),
    dict(shape=(1, 6, 20, 28), pad=5, k=3, md=4, s2=1),            # 3x3 kernel window: sums over up to 9 outputs
])
def test_reference_correlation_backward_equals_oracle_and_product(cfg, request):
    """correlation_cuda.backward of the reference binary (correlation_cuda_kernel.cu:148-333) vs oracle vs product,
    stride1 = 1; fp32 summation order differs between the three, so compare to 1e-5 relative."""
    ref = _ref("correlation_cuda")
    g = torch.Generator().manual_seed(cfg["shape"][1] + cfg["md"])
    a = torch.randn(cfg["shape"], generator=g).to(DEV)
    b = torch.randn(cfg["shape"], generator=g).to(DEV)
    out = ops.correlation(a, b, cfg["pad"], cfg["k"], cfg["md"], 1, cfg["s2"], 1)
    go = torch.randn(out.shape, generator=g).to(DEV)
    g1 = g2 = None
    if ref is not None:
        r1, r2, g1, g2 = a.new_empty(0), a.new_empty(0), a.new_empty(0), a.new_empty(0)      # correlation.py:37-42
        ref.backward(a, b, r1, r2, go, g1, g2, cfg["pad"], cfg["k"], cfg["md"], 1, cfg["s2"], 1)
        torch.cuda.synchronize()
    got1, got2 = ops.correlation_backward(a, b, go, cfg["pad"], cfg["k"], cfg["md"], 1, cfg["s2"], 1)
    o1, o2 = orc.correlation_backward(a.cpu().numpy(), b.cpu().numpy(), go.cpu().numpy(), cfg["pad"], cfg["k"], cfg["md"], cfg["s2"])
    for k, want, got, o in ((1, g1, got1, o1), (2, g2, got2, o2)):
        case = f"{request.node.name}/grad_input{k}"
        assert np.abs(o).max() > 0
        tol = pin.assert_close(case, o, want)
        pin.assert_close(case, got, want)
        assert np.abs(got.cpu().numpy() - o).max() <= 2 * tol


def test_correlation_function_autograd():
    """CorrelationFunction.backward through autograd against a finite difference of the forward."""
    from video_super_resolution_b200.my_packages.FlowProjection.networks.correlation_package.correlation import Correlation
    g = torch.Generator().manual_seed(3)
    a = torch.randn((1, 4, 12, 16), generator=g).to(DEV).requires_grad_(True)
    b = torch.randn((1, 4, 12, 16), generator=g).to(DEV).requires_grad_(True)
    corr = Correlation(pad_size=4, kernel_size=1, max_displacement=4, stride1=1, stride2=2)
    w = torch.randn(corr(a, b).shape, generator=g).to(DEV)
    (corr(a, b) * w).sum().backward()
    eps = 1e-2
    with torch.no_grad():
        for t, grad in ((a, a.grad), (b, b.grad)):
            base = (corr(a, b) * w).sum()
            t[0, 2, 5, 7] += eps
            num = ((corr(a, b) * w).sum() - base) / eps
            t[0, 2, 5, 7] -= eps
            assert abs(num.item() - grad[0, 2, 5, 7].item()) <= 2e-2 * max(1.0, abs(num.item()))
    with pytest.raises(RuntimeError):
        ops.correlation_backward(a.detach(), b.detach(), w, 4, 1, 4, 2, 2, 1)          # stride1 != 1: unsupported


@pytest.mark.parametrize("ks", [2, 3])
def test_reference_resample2d_kernel_size_gt_1(ks, request):
    """resample2d_kernel.cu:54-61: the taps summed over a ks x ks window with un-clamped NCHW address arithmetic.  Equal to
    the reference binary wherever the reference stays inside its tensor (the last rows of the LAST plane read out of
    bounds there; those outputs are excluded)."""
    ref = _ref("resample2d_cuda")
    B, C, H, W = 2, 3, 40, 56
    g = torch.Generator().manual_seed(ks)
    img = (torch.rand((B, C, H, W), generator=g) * 255).to(DEV)
    flow = ((torch.rand((B, 2, H, W), generator=g) - 0.5) * 10).to(DEV)
    # guard rows after the tensor so that the reference's out-of-bounds reads hit our own allocation, not a fault
    big = torch.zeros((B * C * H + 8, W), device=DEV)
    big[:B * C * H] = img.reshape(-1, W)
    img_v = big[:B * C * H].view(B, C, H, W)
    got = ops.resample2d(img_v, flow, ks, True)
    ok = torch.ones((B, C, H, W), dtype=torch.bool, device=DEV)
    ok[B - 1, C - 1, H - ks - 7:] = False          # |flow| <= 5: taps of these outputs may lie past the end of the tensor
    want = None
    if ref is not None:
        out = torch.zeros_like(img)
        ref.forward(img_v, flow, out, ks, True)
        torch.cuda.synchronize()
        want = out[ok]
    pin.assert_equal(request.node.name, got[ok], want)
    assert (got[ok] - ops.resample2d(img_v, flow, 1, True)[ok]).abs().max().item() > 1.0     # ks really matters
    with pytest.raises(Exception):
        ops.resample2d(img_v, flow, 17, True)


@pytest.mark.parametrize("dtype", [torch.float16, torch.float64])
def test_reference_channelnorm_fp16_fp64(dtype, request):
    """The other dtypes of AT_DISPATCH_FLOATING_TYPES_AND_HALF (channelnorm_kernel.cu:111,152), forward and backward,
    bit for bit against the reference binary."""
    ref = _ref("channelnorm_cuda")
    shape = (2, 3, 37, 50)
    x = (torch.randn(shape, generator=torch.Generator().manual_seed(1)) * 20).to(DEV, dtype)
    gout = torch.randn((shape[0], 1, shape[2], shape[3]), generator=torch.Generator().manual_seed(2)).to(DEV, dtype)
    got = ops.channelnorm(x)
    out = gin = None
    if ref is not None:
        out = torch.zeros((shape[0], 1, shape[2], shape[3]), device=DEV, dtype=dtype)
        ref.forward(x, out, 2)
        gin = torch.zeros_like(x)
        ref.backward(x, out, gout, gin, 2)
        torch.cuda.synchronize()
    assert got.dtype == dtype
    pin.assert_equal(request.node.name + "/forward", got, out)
    pin.assert_equal(request.node.name + "/backward", ops.channelnorm_backward(x, got if out is None else out, gout), gin)
