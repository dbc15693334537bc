"""Drop-in for the reference's pybind module `resample2d_cuda` (resample2d_cuda.cc:6-31), over libvsr_b200.so."""
from ._abi import L, check, stream


def forward(input1, input2, output, kernel_size, bilinear):
    """resample2d_cuda_forward(input1, input2, output, kernel_size, bilinear) -- resample2d.py:21"""
    B, C, H, W = output.shape
    with __import__("torch").cuda.device(output.device):
        return check(L().vsr_resample2d_forward(input1.data_ptr(), input2.data_ptr(), output.data_ptr(), B, C, H, W,
                                                int(kernel_size), int(bool(bilinear)), stream()), "vsr_resample2d_forward")


def backward(input1, input2, grad_output, grad_input1, grad_input2, kernel_size, bilinear):
    """resample2d_cuda_backward(...) -- resample2d.py:35-37; grad_input1 arrives zero-filled (:32).
    Under torch.use_deterministic_algorithms(True) grad_input1 comes from the deterministic kernel (bit-identical to the
    CPU restatement on every run) instead of the atomic scatter, so the reference's Resample2dFunction honours the flag."""
    B, C, H, W = grad_output.shape
    torch = __import__("torch")
    if torch.are_deterministic_algorithms_enabled():
        from .. import ops
        ops._resample2d_backward_into(input1, input2, grad_output, grad_input1, grad_input2, kernel_size, bilinear,
                                      deterministic=True)
        return 1
    with torch.cuda.device(grad_output.device):
        return check(L().vsr_resample2d_backward(input1.data_ptr(), input2.data_ptr(), grad_output.data_ptr(),
                                                 grad_input1.data_ptr(), grad_input2.data_ptr(), B, C, H, W,
                                                 int(kernel_size), int(bool(bilinear)), stream()), "vsr_resample2d_backward")
