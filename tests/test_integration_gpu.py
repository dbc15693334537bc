"""INTEGRATION.md 2, executed: the REFERENCE's own autograd Functions (`Resample2d`, `ChannelNorm`, `Correlation`:
resample2d.py, channelnorm.py, correlation.py, staged unmodified under oracle/_ref/pyref by oracle/build_ref.py) run
over the drop-in stubs of video_super_resolution_b200/integration/ -- i.e. over libvsr_b200.so -- and are compared with
the same classes running over the reference's own compiled extensions (oracle/_ref/*.so).
Without the reference's files, the calls those classes make into their extension (restated below) run over the same
stubs and are compared with the reference classes' stored outputs (tests/ref_pins.py)."""
import sys
from types import SimpleNamespace

import pytest
import torch

from oracle import build_ref
from tests import ref_pins as pin
from video_super_resolution_b200 import integration

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _ext(name):
    return sys.modules[name + "_cuda"]          # bound like the reference's module-level `import <name>_cuda`


class _Resample2dFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, input1, input2, kernel_size=1, bilinear=True):
        assert input1.is_contiguous() and input2.is_contiguous()                           # resample2d.py:10-11
        ctx.save_for_backward(input1, input2)
        ctx.kernel_size, ctx.bilinear = kernel_size, bilinear
        output = input1.new_zeros(input1.size())                                           # resample2d.py:17-19
        _ext("resample2d").forward(input1, input2, output, kernel_size, bilinear)          # resample2d.py:21
        return output

    @staticmethod
    def backward(ctx, grad_output):
        input1, input2 = ctx.saved_tensors
        grad_input1 = input1.new_zeros(input1.size())                                      # resample2d.py:32
        grad_input2 = input1.new_zeros(input2.size())                                      # resample2d.py:33
        _ext("resample2d").backward(input1, input2, grad_output.contiguous(), grad_input1, grad_input2,
                                    ctx.kernel_size, ctx.bilinear)                         # resample2d.py:35-37
        return grad_input1, grad_input2, None, None


class _Resample2d(torch.nn.Module):
    def __init__(self, kernel_size=1, bilinear=True):
        super().__init__()
        self.kernel_size, self.bilinear = kernel_size, bilinear

    def forward(self, input1, input2):
        return _Resample2dFunction.apply(input1.contiguous(), input2, self.kernel_size, self.bilinear)   # :48-51


class _ChannelNormFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, input1, norm_deg=2):
        assert input1.is_contiguous()
        b, _, h, w = input1.size()
        output = input1.new_zeros((b, 1, h, w))
        _ext("channelnorm").forward(input1, output, norm_deg)                              # channelnorm.py:14
        ctx.save_for_backward(input1, output)
        ctx.norm_deg = norm_deg
        return output

    @staticmethod
    def backward(ctx, grad_output):
        input1, output = ctx.saved_tensors
        grad_input1 = input1.new_zeros(input1.size())
        _ext("channelnorm").backward(input1, output, grad_output, grad_input1, ctx.norm_deg)   # channelnorm.py:26-27
        return grad_input1, None


class _ChannelNorm(torch.nn.Module):
    def __init__(self, norm_deg=2):
        super().__init__()
        self.norm_deg = norm_deg

    def forward(self, input1):
        return _ChannelNormFunction.apply(input1, self.norm_deg)                          # channelnorm.py:32-39


class _CorrelationFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, input1, input2, args):
        ctx.save_for_backward(input1, input2)
        ctx.args = args
        rbot1, rbot2, output = input1.new_empty(0), input2.new_empty(0), input1.new_empty(0)     # correlation.py:22-24
        _ext("correlation").forward(input1, input2, rbot1, rbot2, output, *args)              # correlation.py:26-28
        return output

    @staticmethod
    def backward(ctx, grad_output):
        input1, input2 = ctx.saved_tensors
        rbot1, rbot2 = input1.new_empty(0), input2.new_empty(0)                                   # correlation.py:37-42
        grad_input1, grad_input2 = input1.new_empty(0), input2.new_empty(0)
        _ext("correlation").backward(input1, input2, rbot1, rbot2, grad_output, grad_input1, grad_input2,
                                     *ctx.args)                                                  # correlation.py:42-45
        return grad_input1, grad_input2, None


class _Correlation(torch.nn.Module):
    def __init__(self, pad_size=0, kernel_size=0, max_displacement=0, stride1=1, stride2=2, corr_multiply=1):
        super().__init__()
        self.args = (pad_size, kernel_size, max_displacement, stride1, stride2, corr_multiply)

    def forward(self, input1, input2):
        return _CorrelationFunction.apply(input1, input2, self.args)


# the reference wrappers' calls into their extension, for when the wrapper files themselves are absent
_CALLS = SimpleNamespace(Resample2d=_Resample2d, ChannelNorm=_ChannelNorm, Correlation=_Correlation)


def _wrapper(name, backend):
    """The reference's wrapper module `name`.py bound to `backend` in {"b200", "reference"}.  Without the reference's
    files: the restated calls over the stubs for "b200", None for "reference" (its outputs are pinned)."""
    ext = name + "_cuda"
    if backend == "b200":
        integration.install()
        w = build_ref.load_py(name)
        return _CALLS if w is None else w
    mod = build_ref.load_ref(ext)
    if mod is None or build_ref.load_py(name) is None:
        return None
    sys.modules[ext] = mod
    return build_ref.load_py(name)


def _run_both(name, run):
    """(b200 results, reference results or Nones when the reference's files are absent)."""
    b200 = run(_wrapper(name, "b200"))
    ref = _wrapper(name, "reference")
    return b200, (run(ref) if ref is not None else (None,) * len(b200))


def test_reference_resample2d_class_over_the_stub():
    g = torch.Generator().manual_seed(3)
    img = (torch.rand((2, 3, 40, 56), generator=g) * 255).to(DEV)
    flow = ((torch.rand((2, 2, 40, 56), generator=g) - 0.5) * 12).to(DEV)
    gout = torch.randn((2, 3, 40, 56), generator=g).to(DEV)

    def run(w):
        a, f = img.clone().requires_grad_(True), flow.clone().requires_grad_(True)
        out = w.Resample2d()(a, f)                          # resample2d.py:42-51 -> Resample2dFunction.apply
        out.backward(gout)
        nearest = w.Resample2d(bilinear=False)(img, flow)
        return out.detach().cpu().numpy(), a.grad.cpu().numpy(), f.grad.cpu().numpy(), nearest.cpu().numpy()
    got, want = _run_both("resample2d", run)
    name = "test_reference_resample2d_class_over_the_stub"
    pin.assert_equal(name + "/forward", got[0], want[0])                    # forward: bit for bit
    pin.assert_equal(name + "/nearest", got[3], want[3])                    # nearest: bit for bit
    pin.assert_equal(name + "/grad_flow", got[2], want[2])                  # flow gradient: bit for bit
    pin.assert_close(name + "/grad_input", got[1], want[1], rel=1e-4)       # input gradient: fp32 atomic order


def test_reference_channelnorm_class_over_the_stub():
    x = (torch.randn((2, 3, 33, 47), generator=torch.Generator().manual_seed(1)) * 20).to(DEV)
    gout = torch.randn((2, 1, 33, 47), generator=torch.Generator().manual_seed(2)).to(DEV)

    def run(w):
        a = x.clone().requires_grad_(True)
        out = w.ChannelNorm()(a)                            # channelnorm.py:32-39
        out.backward(gout)
        return out.detach().cpu().numpy(), a.grad.cpu().numpy()
    got, want = _run_both("channelnorm", run)
    pin.assert_equal("test_reference_channelnorm_class_over_the_stub/forward", got[0], want[0])
    pin.assert_equal("test_reference_channelnorm_class_over_the_stub/grad_input", got[1], want[1])


def test_reference_correlation_class_over_the_stub():
    g = torch.Generator().manual_seed(5)
    a0 = torch.randn((1, 16, 24, 32), generator=g).to(DEV)
    b0 = torch.randn((1, 16, 24, 32), generator=g).to(DEV)

    def run(w):
        a, b = a0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
        # FlowNetC's configuration (FlowNetC.py:22)
        out = w.Correlation(pad_size=20, kernel_size=1, max_displacement=20, stride1=1, stride2=2, corr_multiply=1)(a, b)
        gout = torch.randn(out.shape, generator=torch.Generator().manual_seed(7)).to(DEV)
        out.backward(gout)
        return out.detach().cpu().numpy(), a.grad.cpu().numpy(), b.grad.cpu().numpy()
    got, want = _run_both("correlation", run)
    for k, part in enumerate(("forward", "grad_input1", "grad_input2")):                # fp32 summation order
        pin.assert_close(f"test_reference_correlation_class_over_the_stub/{part}", got[k], want[k])
