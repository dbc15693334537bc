"""CPU: the host logic of the map-parallel path (one window over a map group, DESIGN.md 11) -- map and band partitions,
the all_to_all split sizes against the pack layout, map-group construction, argument checks of the C ABI (no kernel
runs here), and the refusal of a gloo group."""
import ctypes
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from video_super_resolution_b200 import _lib
from video_super_resolution_b200.map_parallel import (MapGroup, band_bounds, exchange_splits, map_group_ranks,
                                                      map_ranges, new_map_groups)


@pytest.mark.parametrize("M", [2, 8, 14, 20, 64])
def test_map_ranges_cover_all_maps_once_balanced(M):
    for G in range(1, M + 1):
        rs = map_ranges(M, G)
        assert len(rs) == G and rs[0][0] == 0 and rs[-1][1] == M
        assert all(rs[r][1] == rs[r + 1][0] for r in range(G - 1))          # contiguous, in rank order
        sizes = [b - a for a, b in rs]
        assert min(sizes) >= 1 and max(sizes) - min(sizes) <= 1
    assert [b - a for a, b in map_ranges(20, 8)] == [3, 3, 3, 3, 2, 2, 2, 2]


def test_map_ranges_reject_more_ranks_than_maps():
    with pytest.raises(ValueError):
        map_ranges(8, 9)
    with pytest.raises(ValueError):
        map_ranges(8, 0)


@pytest.mark.parametrize("h", [1, 7, 9, 64, 270, 360])
@pytest.mark.parametrize("s", [2, 4])
def test_band_bounds_cover_rows_at_lr_row_boundaries(h, s):
    for G in range(1, min(h, 8) + 1):
        lb = band_bounds(h, G)
        assert len(lb) == G + 1 and lb[0] == 0 and lb[-1] == h
        sizes = [lb[p + 1] - lb[p] for p in range(G)]
        assert min(sizes) >= 1 and max(sizes) - min(sizes) <= 1
        W = s * 5
        for p in range(G):
            rows = s * sizes[p]
            # HR band = whole LR rows; every map plane of a band (3*rows*W floats) keeps the fc's float4 loads aligned
            # and its 4 outputs per thread inside one channel (rows*W % 4 == 0)
            assert (s * lb[p]) % s == 0 and (3 * rows * W) % 4 == 0 and (rows * W) % 4 == 0
    with pytest.raises(ValueError):
        band_bounds(3, 4)


@pytest.mark.parametrize("M,h,w,s", [(8, 9, 5, 4), (20, 270, 480, 4), (14, 7, 3, 2), (8, 360, 720, 4)])
def test_exchange_splits_match_pack_layout(M, h, w, s):
    for G in range(1, min(M, h, 8) + 1):
        maps, lb = map_ranges(M, G), band_bounds(h, G)
        H, W = s * h, s * w
        splits = [exchange_splits(M, h, w, s, G, r) for r in range(G)]
        for r in range(G):
            send, recv = splits[r]
            nmaps = maps[r][1] - maps[r][0]
            # pack: band p of rank r's maps (nmaps,3,rows_p,W), back to back; starts at nmaps*3*s*l_p*W floats
            assert sum(send) == nmaps * 3 * H * W
            assert all(sum(send[:p]) == nmaps * 3 * s * lb[p] * W for p in range(G))
            rows = s * (lb[r + 1] - lb[r])
            assert sum(recv) == M * 3 * rows * W                                 # (M,3,rows,W) in map order
            assert all(sum(recv[:q]) == maps[q][0] * 3 * rows * W for q in range(G))
            for q in range(G):
                assert send[q] == splits[q][1][r]                               # what r sends q is what q expects


def test_map_group_ranks():
    assert map_group_ranks(8, 2) == [[0, 1], [2, 3], [4, 5], [6, 7]]
    assert map_group_ranks(8, 8) == [list(range(8))]
    assert map_group_ranks(4, 1) == [[0], [1], [2], [3]]
    with pytest.raises(ValueError):
        map_group_ranks(6, 4)


def _plan(M=8, h=9, w=5, scale=4):
    L = _lib.lib()
    cfg = _lib.SrfbnConfig(M, h, w, 3, 6, 32, scale)
    plan = ctypes.c_void_p()
    assert L.vsr_srfbn_plan_create(ctypes.byref(cfg), ctypes.byref(plan)) == 0
    return L, plan


def test_plan_map_range_arguments():
    L, plan = _plan(M=20)
    try:
        full = L.vsr_srfbn_workspace_bytes(plan)
        assert L.vsr_srfbn_plan_set_map_range(plan, 3, 3) == 1
        assert L.vsr_srfbn_plan_set_map_range(plan, -1, 3) == 1
        assert L.vsr_srfbn_plan_set_map_range(plan, 0, 21) == 1
        assert L.vsr_srfbn_plan_set_map_range(plan, 6, 9) == 0
        assert L.vsr_srfbn_chunk_maps(plan) == 3
        assert L.vsr_srfbn_workspace_bytes(plan) < full                          # per-map images of 3 maps, not 20
        assert L.vsr_srfbn_plan_set_windows(plan, 2) == 2                        # windows > 1 with a range: unsupported
        assert L.vsr_srfbn_plan_set_windows(plan, 1) == 0
        # a workspace cap chunks inside the range: the chunk is a divisor of the range's 3 maps
        one = L.vsr_srfbn_workspace_bytes(plan)
        assert L.vsr_srfbn_plan_set_workspace_cap(plan, one - 1) == 0
        assert L.vsr_srfbn_chunk_maps(plan) == 1
        # a range no chunk fits under the cap (the per-map images of 20 maps, not 3) leaves the plan as it was
        capped = L.vsr_srfbn_workspace_bytes(plan)
        assert L.vsr_srfbn_plan_set_workspace_cap(plan, capped) == 0
        assert L.vsr_srfbn_plan_set_map_range(plan, 0, 20) == 3
        assert L.vsr_srfbn_chunk_maps(plan) == 1 and L.vsr_srfbn_workspace_bytes(plan) == capped
        # host-side checks of the band entry points run before any CUDA call; an unbound plan is a state error
        b = (ctypes.c_int * 3)(0, 5, 9)
        assert L.vsr_srfbn_pack_bands(plan, b, 2, 1, None) == 4
        assert L.vsr_srfbn_pack_bands(plan, (ctypes.c_int * 3)(0, 5, 8), 2, 1, None) == 1   # does not end at h
        assert L.vsr_srfbn_pack_bands(plan, (ctypes.c_int * 3)(0, 0, 9), 2, 1, None) == 1   # empty band
        assert L.vsr_srfbn_fuse_band(plan, 16, 8, 16, None, None) == 4
        assert L.vsr_srfbn_forward_maps(plan, 16, None) == 4
        assert L.vsr_srfbn_forward_maps_refresh(plan, 16, 7, None) == 4
    finally:
        L.vsr_srfbn_plan_destroy(plan)
    L, plan = _plan()
    try:
        assert L.vsr_srfbn_plan_set_windows(plan, 3) == 0
        assert L.vsr_srfbn_plan_set_map_range(plan, 0, 4) == 2                  # and in the other order
    finally:
        L.vsr_srfbn_plan_destroy(plan)


def test_unpack_bands_arguments():
    L = _lib.lib()
    b = (ctypes.c_int * 3)(0, 3, 5)
    assert L.vsr_unpack_bands(None, 4, 4, 3, 8, b, 2, 0, None) == 1
    assert L.vsr_unpack_bands(4, 4, 2, 3, 8, b, 2, 0, None) == 1                   # elem_bytes 1 or 4
    assert L.vsr_unpack_bands(4, 4, 4, 0, 8, b, 2, 0, None) == 1
    assert L.vsr_unpack_bands(4, 4, 4, 3, 8, (ctypes.c_int * 3)(0, 3, 3), 2, 0, None) == 1
    assert L.vsr_unpack_bands(4, 4, 4, 3, 8, b, 65, 0, None) == 1
    assert L.vsr_unpack_bands(4, 4, 4, 3, 8, b, 2, 3 * 3 * 8 - 1, None) == 1        # a band does not fit its stride
    assert L.vsr_unpack_bands(6, 4, 4, 3, 8, b, 2, 0, None) == 1                   # misaligned for 4-byte elements


def _fake(size, rank=0):
    class Fake:
        pass
    g = Fake()
    g.size, g.rank = size, rank
    g.broadcast = g.all_to_all = g.all_gather = None
    return g


def test_module_and_pipeline_reject_bad_groups():
    from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
    from video_super_resolution_b200.pipeline import WarpFusePipeline
    with pytest.raises(ValueError):
        SRProjectionModule(num_maps=8, map_group=_fake(9))                      # G > M
    sr = SRProjectionModule(num_maps=8, map_group=_fake(2))
    with pytest.raises(ValueError, match="windows"):
        WarpFusePipeline(3, 9, 5, sr, device="cpu", windows=2, map_group=sr.map_group)
    with pytest.raises(ValueError, match="same map_group"):
        WarpFusePipeline(3, 9, 5, SRProjectionModule(num_maps=8), device="cpu", map_group=sr.map_group)
    with pytest.raises(ValueError, match="same map_group"):
        WarpFusePipeline(3, 9, 5, sr, device="cpu")


def test_gloo_group_is_refused():
    store = dist.HashStore()
    dist.init_process_group("gloo", store=store, rank=0, world_size=1)
    try:
        with pytest.raises(ValueError, match="gloo"):
            MapGroup(dist.group.WORLD)
        from video_super_resolution_b200.my_packages.SRProjection.SRProjectionModule import SRProjectionModule
        with pytest.raises(ValueError, match="NCCL"):
            SRProjectionModule(num_maps=8, map_group=dist.group.WORLD)
    finally:
        dist.destroy_process_group()


def _groups_worker(rank, world, G, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        idx, pg, n = new_map_groups(G)
        ranks = dist.get_process_group_ranks(pg)
        t = torch.tensor([rank], dtype=torch.int64)
        dist.all_reduce(t, group=pg)                       # the group holds exactly its ranks
        out[rank] = (idx, n, ranks, int(t))
    finally:
        dist.destroy_process_group()


def test_new_map_groups_world4_gloo():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_groups_worker, args=(4, 2, port, out), nprocs=4, join=True)
    assert dict(out) == {0: (0, 2, [0, 1], 1), 1: (0, 2, [0, 1], 1), 2: (1, 2, [2, 3], 5), 3: (1, 2, [2, 3], 5)}
