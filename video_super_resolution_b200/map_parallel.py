"""One frame window over the G GPUs of a map group (DESIGN.md 11).

The M = 3T-1 maps of a window go through the conv stack independently until the per-pixel fc, which needs all M maps
of a pixel and nothing of any other pixel.  So rank r of a map group convolves the maps `map_ranges(M, G)[r]`, the
ranks exchange row bands of the per-map images with one all_to_all, and rank p fuses the HR rows of its band
`band_bounds(h, G)` -- with the same kernels and the same additions as one GPU, so every output pixel is bit-identical.

A map group is a torch.distributed process group of NCCL ranks, one GPU each.  `MapGroup` is the handful of
collectives the map-parallel path issues on it; the module and the pipeline call nothing else, so a stand-in with
the same four methods can run the partition and exchange of G ranks on one device.
"""
from __future__ import annotations


def map_ranges(M: int, G: int) -> list:
    """[(m_r, m_{r+1})] for r < G: [0, M) in G contiguous ranges in rank order, sizes differing by at most 1 (the
    first M % G ranks take one more map)."""
    if G < 1 or G > M:
        raise ValueError(f"a map group of {G} ranks cannot split {M} maps (1 <= G <= M)")
    q, rem = divmod(M, G)
    out, m = [], 0
    for r in range(G):
        n = q + (r < rem)
        out.append((m, m + n))
        m += n
    return out


def band_bounds(h: int, G: int) -> list:
    """LR row boundaries 0 = l_0 < l_1 < ... < l_G = h of the G row bands (sizes differing by at most 1).  Band p is the
    HR rows [s*l_p, s*l_{p+1}): whole LR rows, so that its estimate slot is a band of LR rows and every map plane of it
    is a multiple of s*s*3 floats -- 16-byte aligned for the fc kernel's 4-float loads, with no ragged tail."""
    if G < 1 or G > h:
        raise ValueError(f"a map group of {G} ranks cannot split {h} LR rows into bands (1 <= G <= h)")
    q, rem = divmod(h, G)
    out = [0]
    for p in range(G):
        out.append(out[-1] + q + (p < rem))
    return out


def exchange_splits(M: int, h: int, w: int, scale: int, G: int, rank: int):
    """(input_split_sizes, output_split_sizes) in floats of the all_to_all of `rank`: it sends band p of its maps to rank
    p and receives band `rank` of rank q's maps from rank q."""
    maps, lb = map_ranges(M, G), band_bounds(h, G)
    W = scale * w
    mine = maps[rank][1] - maps[rank][0]
    rows = [scale * (lb[p + 1] - lb[p]) for p in range(G)]
    send = [mine * 3 * rows[p] * W for p in range(G)]
    recv = [(maps[q][1] - maps[q][0]) * 3 * rows[rank] * W for q in range(G)]
    return send, recv


def map_group_ranks(world: int, G: int) -> list:
    """The ranks of each map group when `world` = groups x G ranks are split into groups of G consecutive ranks."""
    if G < 1 or world % G:
        raise ValueError(f"a world of {world} ranks does not split into map groups of {G}")
    return [list(range(g * G, (g + 1) * G)) for g in range(world // G)]


def new_map_groups(G: int):
    """Splits the default process group into groups of G consecutive ranks (every rank must call this).  Returns
    (this rank's group index, its process group, number of groups).  Shard the chunks of a video over the groups with
    pipeline.shard_chunks(chunks, num_groups, index) and run each group's chunks with run_sequence(map_group=pg)."""
    import torch.distributed as dist
    world, rank = dist.get_world_size(), dist.get_rank()
    groups = map_group_ranks(world, G)
    mine = None
    for g, ranks in enumerate(groups):
        pg = dist.new_group(ranks)                     # collective: every rank creates every group, in the same order
        if rank in ranks:
            mine = (g, pg)
    return mine[0], mine[1], len(groups)


class MapGroup:
    """The collectives of the map-parallel path on an NCCL process group (one GPU per rank)."""

    def __init__(self, pg):
        import torch.distributed as dist
        if not dist.is_available() or not dist.is_initialized():
            raise RuntimeError("map_group: torch.distributed is not initialised")
        backend = str(dist.get_backend(pg)).lower()
        if "nccl" not in backend:
            raise ValueError(f"map_group: the map-parallel path exchanges device buffers over NCCL; a {backend!r} "
                             "group (CPU / gloo) is not supported")
        self.pg = pg
        self.rank = dist.get_rank(pg)
        self.size = dist.get_world_size(pg)

    def broadcast(self, t, src: int = 0):
        """t from group rank src to every rank, in place."""
        import torch.distributed as dist
        dist.broadcast(t, group_src=src, group=self.pg)

    def all_to_all(self, out, inp, out_splits, in_splits):
        import torch.distributed as dist
        dist.all_to_all_single(out, inp, output_split_sizes=out_splits, input_split_sizes=in_splits, group=self.pg)

    def all_gather(self, out, inp):
        """out (G * inp.numel(),) <- every rank's inp, in rank order."""
        import torch.distributed as dist
        dist.all_gather_into_tensor(out, inp, group=self.pg)


def as_map_group(g):
    """A MapGroup for a process group; an object that already has the MapGroup methods is taken as it is."""
    if g is None or all(hasattr(g, a) for a in ("rank", "size", "broadcast", "all_to_all", "all_gather")):
        return g
    return MapGroup(g)
