"""CPU: the window-batched entry points validate their arguments on the host before any CUDA call, and a plan's
workspace and chunking follow the window count (no compute: there is no GPU here)."""
import ctypes

import pytest

from video_super_resolution_b200 import _lib
from video_super_resolution_b200.pipeline import _runs

INVALID, UNSUPPORTED, WORKSPACE, STATE = 1, 2, 3, 4


def _plan(M=8, h=16, w=24, scale=4):
    L = _lib.lib()
    cfg = _lib.SrfbnConfig(M, h, w, 3, 6, 32, scale)
    plan = ctypes.c_void_p()
    assert L.vsr_srfbn_plan_create(ctypes.byref(cfg), ctypes.byref(plan)) == 0
    return plan


def test_front_entry_points_refuse_bad_window_counts():
    L = _lib.lib()
    # device pointers stand in as 16 (never dereferenced: every call below fails its checks first)
    p = 16
    for nw in (0, -1, 65536):
        assert L.vsr_warp_windows_nhwc3(p, p, p, p, nw, 3, 1, 8, 8, 2, None) == INVALID
        assert L.vsr_assemble_stack_windows(p, p, p, p, p, None, p, p, nw, 0, 3, 1, 8, 8, None) == INVALID
        assert L.vsr_estimate_slot_windows(p, None, p, nw, 0, 8, 8, 4, None) == INVALID
        assert L.vsr_compose_flow_windows(p, p, p, nw, 0, 8, 8, None) == INVALID
        assert L.vsr_warp_labels_u8_windows(p, p, p, nw, 0, 8, 8, None) == INVALID
    for nw in (0, -1):
        assert L.vsr_vos_threshold_windows(p, p, p, nw, 8, 8, None) == INVALID
    # negative or odd strides
    assert L.vsr_assemble_stack_windows(p, p, p, p, p, None, p, p, 2, -1, 3, 1, 8, 8, None) == INVALID
    assert L.vsr_estimate_slot_windows(p, None, p, 2, -3, 8, 8, 4, None) == INVALID
    assert L.vsr_compose_flow_windows(p, p, p, 2, 3, 8, 8, None) == INVALID
    assert L.vsr_warp_labels_u8_windows(p, p, p, 2, 7, 8, 8, None) == INVALID
    # the per-window limits hold as well
    assert L.vsr_warp_windows_nhwc3(p, p, p, p, 2, 3, 3, 8, 8, 2, None) == INVALID      # centre outside 0..T-1


def test_plan_windows_scale_the_workspace_and_chunking():
    L = _lib.lib()
    M = 8
    one, two = _plan(M), _plan(M)
    try:
        assert L.vsr_srfbn_plan_set_windows(two, 0) == INVALID
        assert L.vsr_srfbn_plan_set_windows(two, 65536) == INVALID
        assert L.vsr_srfbn_plan_set_windows(two, 2) == 0
        assert L.vsr_srfbn_chunk_maps(one) == M and L.vsr_srfbn_chunk_maps(two) == 2 * M
        b1, b2 = L.vsr_srfbn_workspace_bytes(one), L.vsr_srfbn_workspace_bytes(two)
        assert 1.9 * b1 < b2 <= 2 * b1 + 64 * 1024
        assert L.vsr_srfbn_weight_bytes(one) == L.vsr_srfbn_weight_bytes(two)     # fc in-features stay M
        # a cap: the largest divisor of W*M that fits, whichever setter comes first
        assert L.vsr_srfbn_plan_set_workspace_cap(two, b1) == 0
        c = L.vsr_srfbn_chunk_maps(two)
        assert c <= M and (2 * M) % c == 0 and L.vsr_srfbn_workspace_bytes(two) <= b1
        assert L.vsr_srfbn_plan_set_windows(two, 3) == 0
        c3 = L.vsr_srfbn_chunk_maps(two)
        assert (3 * M) % c3 == 0 and L.vsr_srfbn_workspace_bytes(two) <= b1
        # a cap no chunk fits under leaves the plan as it was, and the setters after it are held to it
        assert L.vsr_srfbn_plan_set_workspace_cap(two, 0) == 0 and L.vsr_srfbn_chunk_maps(two) == 3 * M
        b3 = L.vsr_srfbn_workspace_bytes(two)
        assert L.vsr_srfbn_plan_set_workspace_cap(two, 1) == WORKSPACE
        assert L.vsr_srfbn_plan_set_windows(two, 2) == WORKSPACE
        assert L.vsr_srfbn_chunk_maps(two) == 3 * M and L.vsr_srfbn_workspace_bytes(two) == b3
        # refresh and forward before bind
        assert L.vsr_srfbn_prepare_refresh(two, 3) == STATE
    finally:
        L.vsr_srfbn_plan_destroy(one)
        L.vsr_srfbn_plan_destroy(two)
    assert L.vsr_srfbn_plan_set_windows(None, 2) == INVALID


def test_runs_of_consecutive_windows():
    assert _runs([]) == []
    assert _runs(range(4)) == [(0, 4)]
    assert _runs([0, 2, 3, 5]) == [(0, 1), (2, 4), (5, 6)]


def test_pipeline_refuses_bad_window_counts_before_touching_the_device():
    from video_super_resolution_b200.pipeline import WarpFusePipeline, run_sequence
    for nw in (0, -2, 1.5):
        with pytest.raises(ValueError):
            WarpFusePipeline(3, 8, 8, device="cpu", windows=nw)
        with pytest.raises(ValueError):
            run_sequence(None, None, None, None, None, [], windows=nw)
