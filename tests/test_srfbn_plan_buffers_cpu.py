"""CPU: the workspace layout vsr_srfbn_debug_buffer reports for created, unbound plans (the buffers the plan walk of
test_srfbn_plan_walk_gpu.py reads), and the argument checks of vsr_srfbn_debug_run_layers, which come before any CUDA
call."""
import ctypes
import os
import re

import pytest

from tests import srfbn_hooks as hk
from video_super_resolution_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, INVALID_ARG, UNSUPPORTED, STATE = 0, 1, 2, 4
NAMES = ["A0", "C128", "XFEAT", "HIDDEN", "LR", "U", "HR", "HB", "HT", "ACC", "PREMIX"]


def test_buffer_ids_are_the_headers():
    text = open(os.path.join(ROOT, "include", "vsr_b200.h")).read()
    ids = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define VSR_SRFBN_BUF_(\w+) (\d+)", text)}
    assert ids == {n: getattr(hk, "BUF_" + n) for n in NAMES}
    assert int(re.search(r"#define VSR_SRFBN_BUFFERS (\d+)", text).group(1)) == len(NAMES)


def _plan(M, h, w, scale, cap_frac=None):
    L = _lib.lib()
    cfg = _lib.SrfbnConfig(M, h, w, 3, 6, 32, scale)
    plan = ctypes.c_void_p()
    _lib.check(L.vsr_srfbn_plan_create(ctypes.byref(cfg), ctypes.byref(plan)), "plan_create")
    if cap_frac is not None:
        full = int(L.vsr_srfbn_workspace_bytes(plan))
        _lib.check(L.vsr_srfbn_plan_set_workspace_cap(plan, int(full * cap_frac)), "set_workspace_cap")
    return plan


def _buffer(plan, id, index):
    off, n = ctypes.c_size_t(), ctypes.c_size_t()
    rc = _lib.lib().vsr_srfbn_debug_buffer(plan, id, index, ctypes.byref(off), ctypes.byref(n))
    return rc, off.value, n.value


@pytest.mark.parametrize("scale", [4, 2])
@pytest.mark.parametrize("cap_frac,chunk", [(None, 6), (0.75, 3), (0.45, 2), (0.22, 1)])
def test_buffers_lie_in_the_workspace_disjoint_and_sized_by_the_chunk(scale, cap_frac, chunk):
    M, h, w = 6, 17, 26
    L = _lib.lib()
    plan = _plan(M, h, w, scale, cap_frac)
    try:
        assert L.vsr_srfbn_chunk_maps(plan) == chunk
        ws = int(L.vsr_srfbn_workspace_bytes(plan))
        P, s2 = chunk * h * w, scale * scale
        lr = P * 64
        size = {hk.BUF_A0: lr, hk.BUF_C128: P * 256, hk.BUF_XFEAT: lr, hk.BUF_HIDDEN: lr, hk.BUF_LR: lr,
                hk.BUF_U: lr, hk.BUF_HB: s2 * P * 64, hk.BUF_PREMIX: M * h * w * s2 * 3 * 4,
                hk.BUF_HR: 4 * P * 64 if scale == 2 else chunk * (h + 1) * (w + 1) * 16 * 64}
        size.update({hk.BUF_HT: 4 * P * 64} if scale == 2 else {hk.BUF_ACC: P * 512})
        missing = {(hk.BUF_ACC, 0)} if scale == 2 else {(hk.BUF_HR, 5), (hk.BUF_HT, 0)}
        spans = []
        for id in range(len(NAMES)):
            for index in range({hk.BUF_LR: 7, hk.BUF_HR: 6}.get(id, 1)):
                rc, off, n = _buffer(plan, id, index)
                if (id, index) in missing:
                    assert rc == UNSUPPORTED, (NAMES[id], index, rc)
                    continue
                assert rc == OK, (NAMES[id], index, rc)
                assert n == size[id], (NAMES[id], index, n, size[id])
                assert off % 1024 == 0 and off + n <= ws, (NAMES[id], index, off, n, ws)
                spans.append((off, off + n, f"{NAMES[id]}[{index}]"))
        assert len(spans) == 7 + 6 + 9 - len(missing)
        spans.sort()
        for (_, end, a), (start, _, b) in zip(spans, spans[1:]):
            assert end <= start, (a, b)
    finally:
        L.vsr_srfbn_plan_destroy(plan)


# What each full-size case of hk.FULL_SIZE_PLANS exists to reach: its largest activation buffer over 2^k bytes, or over
# 2^k BF16 elements (2^(k+1) bytes)
_REACH = {"C2": ("bytes", 31), "C4": ("BF16 elements", 31), "C5-W3": ("bytes", 32), "C2-W2": ("bytes", 32)}


@pytest.mark.parametrize("name", list(hk.FULL_SIZE_PLANS))
def test_full_size_cases_reach_their_sizes(name):
    """The plans of the full-size GPU tests, created as those tests create them, still reach the sizes they exist for:
    a buffer past 2^31 bytes (C2), 2^31 BF16 elements (C4) or 2^32 bytes (the uncapped window-batched cases), and for
    the capped C5 W = 3 case a chunk of maps that straddles window boundaries."""
    M, h, w, scale, W, cap = hk.FULL_SIZE_PLANS[name]
    L = _lib.lib()
    plan = _plan(M, h, w, scale)
    try:
        if W > 1:
            _lib.check(L.vsr_srfbn_plan_set_windows(plan, W), "set_windows")
        if cap is not None:
            _lib.check(L.vsr_srfbn_plan_set_workspace_cap(plan, cap), "set_workspace_cap")
        chunk = L.vsr_srfbn_chunk_maps(plan)
        largest = max(_buffer(plan, id, 0)[2] for id in range(len(NAMES)))
        print(f"[measure] {name}: chunk {chunk}, workspace {L.vsr_srfbn_workspace_bytes(plan) / 2**30:.2f} GiB, "
              f"largest buffer {largest / 2**30:.2f} GiB")
        if cap is None:
            assert chunk == W * M, chunk
        else:
            assert chunk % M and M % chunk and chunk < W * M, chunk             # a chunk straddles the windows
        if name in _REACH:
            unit, k = _REACH[name]
            assert largest > 2 ** (k + (unit != "bytes")), (name, largest, unit, k)
    finally:
        L.vsr_srfbn_plan_destroy(plan)


def test_argument_errors():
    L = _lib.lib()
    plan = _plan(3, 5, 7, 4)
    try:
        for id, index in ((-1, 0), (len(NAMES), 0), (hk.BUF_LR, 7), (hk.BUF_HR, 6), (hk.BUF_A0, 1), (hk.BUF_LR, -1)):
            assert _buffer(plan, id, index)[0] == INVALID_ARG, (id, index)
        n = ctypes.c_size_t()
        assert L.vsr_srfbn_debug_buffer(None, 0, 0, ctypes.byref(n), ctypes.byref(n)) == INVALID_ARG
        assert L.vsr_srfbn_debug_buffer(plan, 0, 0, None, ctypes.byref(n)) == INVALID_ARG
        assert L.vsr_srfbn_debug_buffer(plan, 0, 0, ctypes.byref(n), None) == INVALID_ARG
        # x is a stand-in pointer, never dereferenced: the checks come first
        assert L.vsr_srfbn_debug_run_layers(plan, 1, 0, 1, None) == STATE          # not bound
        assert L.vsr_srfbn_debug_run_layers(plan, None, 0, 1, None) == INVALID_ARG
        assert L.vsr_srfbn_debug_run_layers(None, 1, 0, 1, None) == INVALID_ARG
    finally:
        L.vsr_srfbn_plan_destroy(plan)
