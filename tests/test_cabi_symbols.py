"""CPU: the C-ABI library builds, loads, and exports every function include/vsr_b200.h declares
(no compute calls -- there is no GPU here)."""
import ctypes
import os
import re
import subprocess

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
    """The library is built one way only and reads one environment variable, VSR_CORR_GENERIC (it chooses between two
    live correlation kernels): no switch changes which conv-stack kernels a process runs, no source carries a
    compile-time experiment switch, and the library exports no entry point the header does not declare."""
    from video_super_resolution_b200 import build
    path = build.build()
    with open(path, "rb") as f:
        names = set(re.findall(rb"VSR_[A-Z0-9_]+", f.read()))
    assert names == {b"VSR_CORR_GENERIC"}, sorted(names)

    nm = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\s[TW]\s+(vsr_[a-z0-9_]+)$", nm, flags=re.M))
    assert exported, nm[:2000]
    assert not exported - set(_declared()), sorted(exported - set(_declared()))

    switched = []
    for src in sorted(os.listdir(build.CSRC)):
        text = open(os.path.join(build.CSRC, src)).read()
        switched += [(src, m) for m in sorted(set(re.findall(r"\bVSR_(?:KNOCKOUT|DBG|TRACE)\b", text)))]
    assert not switched, switched


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

    # vsr_test_fused_updown: device pointers stand in as 1 (never dereferenced), weights are real host arrays
    w8 = (ctypes.c_float * (32 * 32 * 64))()
    wt = (ctypes.c_float * (32 * 32 * 6))()
    b = (ctypes.c_float * 32)()
    B, h, w = 2, 5, 7
    need = L.vsr_test_workspace_bytes(B, h, w) + B * h * w * 512

    def updown(nsrc, wu=w8, wd=w8, ws_bytes=need, y=1):
        return L.vsr_test_fused_updown(1, 1, nsrc, 1, B, h, w, wu, b, 0.25, wt, b, 0.3, wd, b, 0.15, y, 1, ws_bytes,
                                       None)
    assert updown(1) == 1 and updown(7) == 1              # nsrc outside 2..6
    assert updown(4, wu=None) == 1 and updown(4, wd=None) == 1 and updown(4, y=None) == 1
    assert updown(2, ws_bytes=need - 1) == 3              # VSR_ERR_WORKSPACE: one byte short of the partial slots
    assert updown(6, ws_bytes=0) == 3


def test_ops_refuse_cpu_tensors():
    import pytest
    import torch
    from video_super_resolution_b200 import ops
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.resample2d(torch.zeros(1, 3, 4, 4), torch.zeros(1, 2, 4, 4))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.project_flow(torch.zeros(1, 4, 4, 2))
