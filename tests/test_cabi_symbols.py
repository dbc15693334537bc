"""CPU: the C-ABI library builds, loads, and exports every function include/vsr_b200.h declares
(no compute calls -- there is no GPU here)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "vsr_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vsr_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from video_super_resolution_b200 import build
    path = build.build()
    lib = ctypes.CDLL(path)
    names = _declared()
    assert len(names) >= 12
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


def test_python_binding_covers_header():
    from video_super_resolution_b200 import _lib
    declared = set(_declared())
    bound = set(_lib.SIGNATURES)
    assert bound <= declared, bound - declared
    assert declared <= bound, declared - bound


def test_shipped_library_reads_no_variant_switches():
    """The shipped library reads one environment variable, VSR_CORR_GENERIC (it chooses between two live correlation
    kernels): no switch changes which conv-stack kernels a process runs.  The timing-experiment switches exist only in
    the -DVSR_KNOCKOUT build."""
    from video_super_resolution_b200 import build
    with open(build.build(), "rb") as f:
        names = set(re.findall(rb"VSR_[A-Z0-9_]+", f.read()))
    assert names == {b"VSR_CORR_GENERIC"}, sorted(names)


def test_host_side_entry_points_without_gpu():
    from video_super_resolution_b200 import _lib
    L = _lib.lib()
    assert b"sm_100a" in L.vsr_version()
    assert L.vsr_error_string(0) == b"ok"
    assert b"workspace" in L.vsr_error_string(3)
    # three rotating cell arrays (16 B per pixel each) + per-image occupancy bitmaps + hole-word lists + flags
    assert 3 * 1080 * 1920 * 16 <= L.vsr_flow_projection_workspace_bytes(8, 1080, 1920) < 3 * 1080 * 1920 * 16 + (8 << 20)
    # argument validation happens before any CUDA call
    assert L.vsr_resample2d_forward(None, None, None, 1, 3, 4, 4, 1, 1, None) == 1
    assert L.vsr_resample2d_forward(1, 1, 1, 1, 3, 4, 4, 17, 1, None) == 2  # kernel_size outside 1..16


def test_ops_refuse_cpu_tensors():
    import pytest
    import torch
    from video_super_resolution_b200 import ops
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.resample2d(torch.zeros(1, 3, 4, 4), torch.zeros(1, 2, 4, 4))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.project_flow(torch.zeros(1, 4, 4, 2))
