"""SRProjectionModule -- the fusion / upsampling convolutions (SRFBN + per-pixel fc over the stacked
maps) with the reference's surface:

    SRProjectionModule(in_channels=3, out_channels=3, num_features=32, upscale_factor=4,
                       num_steps=3, num_groups=6, act_type='prelu', norm_type=None)
    .forward(x (M,3,h,w) fp32 0..255) -> (1,3,s*h,s*w) fp32
    ref: my_packages/SRProjection/SRProjectionModule.py:96-150
    .forward(x (W*M,3,h,w) or (W,M,3,h,w)) -> (W,3,s*h,s*w): W frame windows in one pass of the plan, frame b
    bit-identical to a forward of window b alone
    SRProjectionModule(..., map_group=pg): one window over the G GPUs of an NCCL process group (DESIGN.md 11), every
    frame bit-identical to the one-GPU forward; forward(..., gather=False) returns only this rank's row band

Parameters carry the reference's state-dict names and shapes (SURVEY.md Appendix C), so a
checkpoint written by the reference's main.py:233-237 loads with load_state_dict unchanged; the only
generalisation is `num_maps` (the reference hard-wires fc in-features to 8 = 3*3-1 stacked maps,
:127).  The arithmetic does not run in torch: forward packs the weights to BF16 GEMM operands
(once per weight version) and calls the tcgen05 implicit-GEMM plan of libvsr_b200.so through the
C ABI (vsr_srfbn_*).  The FeedbackBlock follows the INTENDED dense-concat dataflow (Appendix C);
the reference's own forward reads uninitialised memory (:55-59,:70-74).

Inference only (the reference's hot loop runs under no_grad, main.py:199-203): there is no
autograd through the CUDA path.
"""
import ctypes

import torch
import torch.nn as nn

from ... import _lib, ops
from ...map_parallel import as_map_group, band_bounds, exchange_splits, map_ranges

RGB_MEAN = (0.4488, 0.4371, 0.4040)   # SRProjectionModule.py:105
# (kernel, stride, padding) of the up/down projection units.  x4 is the reference's hard-wired geometry
# (SRProjectionModule.py:10-12,101-103); x2 is SRFBN's, needed by BASELINE config C4 (SURVEY.md 8 a6).
GEOMETRY = {4: (8, 4, 2), 2: (6, 2, 2)}


def _block(conv, act=True):
    """ConvBlock / DeconvBlock as nn.Sequential so that parameter names are `<name>.0.weight`,
    `<name>.0.bias`, `<name>.1.weight` (blocks.py:7-43,64-74)."""
    return nn.Sequential(conv, nn.PReLU(num_parameters=1, init=0.2)) if act else nn.Sequential(conv)


class _MeanShift(nn.Conv2d):
    """blocks.py:46-55: frozen 1x1 identity conv with bias sign*255*mean."""

    def __init__(self, rgb_mean, sign=-1):
        super().__init__(3, 3, kernel_size=1)
        self.weight.data = torch.eye(3).view(3, 3, 1, 1)
        self.bias.data = sign * 255.0 * torch.tensor(rgb_mean)
        for p in self.parameters():
            p.requires_grad = False


class _FeedbackParams(nn.Module):
    """Parameter container with FeedbackBlock's names (SRProjectionModule.py:7-42)."""

    def __init__(self, nf, num_groups, ksp=(8, 4, 2)):
        super().__init__()
        self.compress_in = _block(nn.Conv2d(2 * nf, nf, 1))
        self.upBlocks = nn.ModuleList([_block(nn.ConvTranspose2d(nf, nf, *ksp)) for _ in range(num_groups)])
        self.downBlocks = nn.ModuleList([_block(nn.Conv2d(nf, nf, *ksp)) for _ in range(num_groups)])
        self.uptranBlocks = nn.ModuleList([_block(nn.Conv2d(nf * (i + 2), nf, 1)) for i in range(num_groups - 1)])
        self.downtranBlocks = nn.ModuleList([_block(nn.Conv2d(nf * (i + 2), nf, 1)) for i in range(num_groups - 1)])
        self.compress_out = _block(nn.Conv2d(num_groups * nf, nf, 1))


class SRProjectionModule(nn.Module):
    def __init__(self, in_channels=3, out_channels=3, num_features=32, upscale_factor=4, num_steps=3, num_groups=6,
                 act_type='prelu', norm_type=None, num_maps=8, workspace_cap_bytes=None, map_group=None):
        super(SRProjectionModule, self).__init__()
        if (in_channels, out_channels, num_features, num_groups) != (3, 3, 32, 6) \
                or upscale_factor not in GEOMETRY or act_type != 'prelu' or norm_type is not None:
            raise NotImplementedError("the B200 path implements 3->3 channels, 32 features, 6 groups, PReLU, no "
                                      "norm, x4 (k8 s4 p2, the reference's geometry) or x2 (k6 s2 p2)")
        ksp = GEOMETRY[upscale_factor]
        self.num_steps = num_steps
        self.num_features = num_features
        self.upscale_factor = upscale_factor
        self.num_maps = num_maps
        # optional cap on the activation workspace: the plan then processes the maps in chunks (bit-identical results)
        self.workspace_cap_bytes = workspace_cap_bytes
        nf = num_features
        self.sub_mean = _MeanShift(RGB_MEAN, -1)
        self.conv_in = _block(nn.Conv2d(in_channels, 4 * nf, 3, padding=1))
        self.feat_in = _block(nn.Conv2d(4 * nf, nf, 1))
        self.block = _FeedbackParams(nf, num_groups, ksp)
        self.out = _block(nn.ConvTranspose2d(nf, nf, *ksp))
        self.conv_out = _block(nn.Conv2d(nf, out_channels, 3, padding=1), act=False)
        self.add_mean = _MeanShift(RGB_MEAN, 1)
        self.fc = nn.Sequential(nn.Linear(num_maps, 32), nn.ReLU(), nn.Linear(32, 1), nn.ReLU())
        # map_group: an NCCL process group (or a map_parallel.MapGroup); rank r convolves map_ranges(M, G)[r] and fuses
        # the HR rows of band r
        self.map_group = as_map_group(map_group)
        if self.map_group is not None:
            map_ranges(num_maps, self.map_group.size)          # ValueError for G > M
        self._plans = {}          # (M, h, w, device[, W if W > 1][, map range]) -> dict(plan, weights, workspace, version)
        self._keep = []

    # -- C ABI plumbing ---------------------------------------------------------------------------
    def _weights_struct(self):
        """vsr_srfbn_weights over contiguous fp32 host copies of the parameters."""
        keep = []

        def fp(t):
            a = t.detach().to("cpu", torch.float32).contiguous()
            keep.append(a)
            return ctypes.cast(a.data_ptr(), ctypes.POINTER(ctypes.c_float))

        def sl(seq):
            return float(seq[1].weight.detach().reshape(-1)[0])

        W = _lib.SrfbnWeights()
        W.sub_mean_bias, W.add_mean_bias = fp(self.sub_mean.bias), fp(self.add_mean.bias)
        W.conv_in_w, W.conv_in_b, W.conv_in_slope = fp(self.conv_in[0].weight), fp(self.conv_in[0].bias), sl(self.conv_in)
        W.feat_in_w, W.feat_in_b, W.feat_in_slope = fp(self.feat_in[0].weight), fp(self.feat_in[0].bias), sl(self.feat_in)
        b = self.block
        W.compress_in_w, W.compress_in_b, W.compress_in_slope = \
            fp(b.compress_in[0].weight), fp(b.compress_in[0].bias), sl(b.compress_in)
        for i in range(6):
            W.up_w[i], W.up_b[i], W.up_slope[i] = fp(b.upBlocks[i][0].weight), fp(b.upBlocks[i][0].bias), sl(b.upBlocks[i])
            W.down_w[i], W.down_b[i], W.down_slope[i] = \
                fp(b.downBlocks[i][0].weight), fp(b.downBlocks[i][0].bias), sl(b.downBlocks[i])
        for i in range(5):
            W.uptran_w[i], W.uptran_b[i], W.uptran_slope[i] = \
                fp(b.uptranBlocks[i][0].weight), fp(b.uptranBlocks[i][0].bias), sl(b.uptranBlocks[i])
            W.downtran_w[i], W.downtran_b[i], W.downtran_slope[i] = \
                fp(b.downtranBlocks[i][0].weight), fp(b.downtranBlocks[i][0].bias), sl(b.downtranBlocks[i])
        W.compress_out_w, W.compress_out_b, W.compress_out_slope = \
            fp(b.compress_out[0].weight), fp(b.compress_out[0].bias), sl(b.compress_out)
        W.out_w, W.out_b, W.out_slope = fp(self.out[0].weight), fp(self.out[0].bias), sl(self.out)
        W.conv_out_w, W.conv_out_b = fp(self.conv_out[0].weight), fp(self.conv_out[0].bias)
        W.fc0_w, W.fc0_b = fp(self.fc[0].weight), fp(self.fc[0].bias)
        W.fc2_w, W.fc2_b = fp(self.fc[2].weight), fp(self.fc[2].bias)
        return W, keep

    def _version(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def _plan_for(self, M, h, w, device, windows=1, map_range=None):
        # one plan per window count and map range; a one-window plan of all maps keeps the key it has always had
        key = (M, h, w, device.index) + ((windows,) if windows > 1 else ()) + ((map_range,) if map_range else ())
        ent = self._plans.get(key)
        ver = self._version()
        L = _lib.lib()
        if ent is None:
            cfg = _lib.SrfbnConfig(M, h, w, self.num_steps, 6, self.num_features, self.upscale_factor)
            plan = ctypes.c_void_p()
            _lib.check(L.vsr_srfbn_plan_create(ctypes.byref(cfg), ctypes.byref(plan)), "srfbn_plan_create")
            if windows > 1:
                rc = L.vsr_srfbn_plan_set_windows(plan, int(windows))
                if rc:
                    L.vsr_srfbn_plan_destroy(plan)
                    _lib.check(rc, "srfbn_plan_set_windows")
            if map_range:
                rc = L.vsr_srfbn_plan_set_map_range(plan, *map_range)
                if rc:
                    L.vsr_srfbn_plan_destroy(plan)
                    _lib.check(rc, "srfbn_plan_set_map_range")
            if self.workspace_cap_bytes:
                _lib.check(L.vsr_srfbn_plan_set_workspace_cap(plan, int(self.workspace_cap_bytes)), "srfbn_plan_set_workspace_cap")
            ent = {"plan": plan, "version": None, "chunk_maps": int(L.vsr_srfbn_chunk_maps(plan)),
                   "weights": torch.empty(int(L.vsr_srfbn_weight_bytes(plan)), dtype=torch.uint8, device=device),
                   "workspace": torch.empty(int(L.vsr_srfbn_workspace_bytes(plan)), dtype=torch.uint8, device=device)}
            self._plans[key] = ent
        if ent["version"] != ver:
            W, keep = self._weights_struct()
            host = torch.empty(ent["weights"].numel(), dtype=torch.uint8).pin_memory()
            _lib.check(L.vsr_srfbn_pack_weights(ent["plan"], ctypes.byref(W), host.data_ptr()), "srfbn_pack_weights")
            ent["weights"].copy_(host)
            torch.cuda.current_stream(device).synchronize()
            del keep
            _lib.check(L.vsr_srfbn_bind(ent["plan"], ent["weights"].data_ptr(), ent["workspace"].data_ptr(),
                                        ent["workspace"].numel()), "srfbn_bind")
            ent["version"] = ver
            ent["have_premix"] = False          # bind drops the second layer list and the per-map images
            ent["refresh_first"] = None
        return ent

    def _windows_of(self, x):
        """(W*M,3,h,w) or (W,M,3,h,w) -> W; ValueError for any other shape."""
        M = self.num_maps
        if x.dim() == 5 and x.shape[0] >= 1 and tuple(x.shape[1:3]) == (M, 3):
            return x.shape[0]
        if x.dim() == 4 and x.shape[1] == 3 and x.shape[0] >= M and x.shape[0] % M == 0:
            return x.shape[0] // M
        raise ValueError(f"SRProjectionModule: expected ({M},3,h,w), (W*{M},3,h,w) or (W,{M},3,h,w), "
                         f"got {tuple(x.shape)}")

    def forward(self, x, out_u8=None, want_f32=True, changed_from=None, gather=True):
        """x: (M,3,h,w), or W frame windows as (W*M,3,h,w) / (W,M,3,h,w) -> (W,3,s*h,s*w) (W = 1: (1,3,s*h,s*w)).
        out_u8: optional (W,s*h,s*w,3) (W = 1: also (s*h,s*w,3)) u8 CUDA tensor that additionally receives the frames as
        clamp(y,0,255) rounded half to even (the loader's pixel format, utils/video_utils.py:23), written by the fc-fuse
        kernel itself; want_f32=False skips the fp32 frames (then the u8 frames are the only output and are returned).
        changed_from=k: the caller states that, since the previous forward of this module on a stack of this shape, only
        the maps [k, M) of each window changed (the fuse pass, network/video_super_resolution.py:62, feeds the frames
        unchanged): the maps are independent until the per-pixel fc, so only those go through the conv stack again and
        the per-map images of the others are reused -- bit-identical to a full forward.
        With a map group (one window: x (M,3,h,w) or (1,M,3,h,w)): gather=True returns the full frame on every rank (the
        u8 frame all-gathered into out_u8, the fp32 frame (1,3,s*h,s*w) gathered when want_f32); gather=False returns
        this rank's band (1,3,rows,s*w) of the fp32 frame (when want_f32) and writes only the band's rows of out_u8;
        gather="u8" all-gathers the u8 frame into out_u8 and returns the fp32 band (a recurrence that passes the frame
        on as its next estimate needs only its own rows).  Without a map group gather must be True."""
        if not x.is_cuda:
            raise RuntimeError("SRProjectionModule: CUDA tensors only (no CPU fallback)")
        mg = self.map_group
        if mg is None and gather is not True:
            raise ValueError("SRProjectionModule: gather applies to a map group only")
        if gather not in (True, False, "u8"):
            raise ValueError("SRProjectionModule: gather must be True, False or 'u8'")
        nw = self._windows_of(x)
        if mg is not None and nw != 1:
            raise ValueError("SRProjectionModule: a map group runs one frame window per forward (windows > 1 is not "
                             "supported with map_group)")
        x = x.reshape(nw * self.num_maps, *x.shape[-3:])
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.to(torch.float32).contiguous()
        M, h, w = self.num_maps, x.shape[2], x.shape[3]
        s = self.upscale_factor
        shapes = [(nw, s * h, s * w, 3)] + ([(s * h, s * w, 3)] if nw == 1 else [])
        if out_u8 is not None and (not out_u8.is_cuda or out_u8.dtype != torch.uint8 or not out_u8.is_contiguous()
                                   or tuple(out_u8.shape) not in shapes):
            raise ValueError(f"SRProjectionModule: out_u8 must be a contiguous CUDA u8 tensor of shape {shapes[-1]}")
        if out_u8 is None and not want_f32:
            raise ValueError("SRProjectionModule: nothing to compute")
        if mg is not None:
            return self._forward_group(x, out_u8, want_f32, changed_from, gather)
        ent = self._plan_for(M, h, w, x.device, nw)
        y = torch.empty((nw, 3, s * h, s * w), dtype=torch.float32, device=x.device) if want_f32 else None
        L = _lib.lib()
        with torch.cuda.device(x.device):
            yp = y.data_ptr() if y is not None else None
            up = out_u8.data_ptr() if out_u8 is not None else None
            st = torch.cuda.current_stream().cuda_stream
            self._sweep(ent, x, changed_from, lambda: L.vsr_srfbn_forward_u8(ent["plan"], x.data_ptr(), yp, up, st),
                        lambda k: L.vsr_srfbn_forward_refresh_u8(ent["plan"], x.data_ptr(), yp, up, k, st))
        return y if want_f32 else out_u8

    def band_geometry(self, h):
        """(this rank's map range, LR band bounds, HR band bounds) of a map-group forward on LR height h."""
        G, r, s = self.map_group.size, self.map_group.rank, self.upscale_factor
        lb = band_bounds(h, G)
        return map_ranges(self.num_maps, G)[r], lb, [s * b for b in lb]

    def _sweep(self, ent, x, changed_from, full, refresh):
        """The conv stack over this plan's maps: `full` (all maps) or, for changed_from=k, `refresh` (the maps >= k)."""
        L = _lib.lib()
        if changed_from is None or changed_from <= 0:
            _lib.check(full(), "srfbn_forward")
            ent["have_premix"] = True
            return
        if not ent.get("have_premix"):
            raise RuntimeError("SRProjectionModule: changed_from needs a preceding full forward on this shape")
        if ent.get("refresh_first") != int(changed_from):
            _lib.check(L.vsr_srfbn_prepare_refresh(ent["plan"], int(changed_from)), "srfbn_prepare_refresh")
            ent["refresh_first"] = int(changed_from)
        _lib.check(refresh(int(changed_from)), "srfbn_forward_refresh")

    def _forward_group(self, x, out_u8, want_f32, changed_from, gather):
        """forward of one window x (M,3,h,w), checked by forward, over the map group: sweep this rank's maps, pack their
        row bands, one all_to_all, fuse this rank's band, and (gather) all-gather the bands.  Every kernel is the one-GPU
        forward's, on the same values."""
        mg, M, s = self.map_group, self.num_maps, self.upscale_factor
        h, w = x.shape[2], x.shape[3]
        H, W = s * h, s * w
        G, r = mg.size, mg.rank
        (m0, m1), lb, hb = self.band_geometry(h)
        ent = self._plan_for(M, h, w, x.device, 1, (m0, m1))
        rows = [hb[p + 1] - hb[p] for p in range(G)]
        rmax = max(rows)
        if "send" not in ent:          # exchange buffers, sized once per plan
            dev = x.device
            ent["send"] = torch.empty((m1 - m0) * 3 * H * W, dtype=torch.float32, device=dev)
            ent["recv"] = torch.empty(M * 3 * rows[r] * W, dtype=torch.float32, device=dev)
            ent["u8_band"] = torch.empty(rmax * W * 3, dtype=torch.uint8, device=dev)
            ent["u8_all"] = torch.empty(G * rmax * W * 3, dtype=torch.uint8, device=dev)
            ent["splits"] = exchange_splits(M, h, w, s, G, r)
            ent["lb"] = (ctypes.c_int * (G + 1))(*lb)
        L = _lib.lib()
        plan = ent["plan"]
        with torch.cuda.device(x.device):
            st = torch.cuda.current_stream().cuda_stream
            self._sweep(ent, x, changed_from, lambda: L.vsr_srfbn_forward_maps(plan, x.data_ptr(), st),
                        lambda k: L.vsr_srfbn_forward_maps_refresh(plan, x.data_ptr(), k, st))
            _lib.check(L.vsr_srfbn_pack_bands(plan, ent["lb"], G, ent["send"].data_ptr(), st), "srfbn_pack_bands")
            send_splits, recv_splits = ent["splits"]
            mg.all_to_all(ent["recv"], ent["send"], recv_splits, send_splits)
            yb = torch.empty(3 * rmax * W, dtype=torch.float32, device=x.device) if want_f32 else None
            band = yb[:3 * rows[r] * W].view(1, 3, rows[r], W) if want_f32 else None
            if out_u8 is None:
                u8p = None
            elif gather:
                u8p = ent["u8_band"].data_ptr()
            else:
                u8p = out_u8.data_ptr() + hb[r] * W * 3           # this band's rows of the caller's (H,W,3) frame
            _lib.check(L.vsr_srfbn_fuse_band(plan, ent["recv"].data_ptr(), rows[r], yb.data_ptr() if want_f32 else None,
                                             u8p, st), "srfbn_fuse_band")
            if out_u8 is not None and gather:
                mg.all_gather(ent["u8_all"], ent["u8_band"])
                ops.unpack_bands(ent["u8_all"], out_u8, hb, 1, W * 3, rmax * W * 3)
            if gather is not True:
                return band if want_f32 else out_u8
            if not want_f32:
                return out_u8
            y_all = torch.empty(G * yb.numel(), dtype=torch.float32, device=x.device)
            mg.all_gather(y_all, yb)
            y = torch.empty((1, 3, H, W), dtype=torch.float32, device=x.device)
            return ops.unpack_bands(y_all, y, hb, 3, W, yb.numel())

    def premix(self, x):
        """Test hook: per-map outputs before the fc fuse, (W*M,3,s*h,s*w) (SRProjectionModule.py:143)."""
        self.forward(x)
        nw = self._windows_of(x)
        M, h, w = self.num_maps, x.shape[-2], x.shape[-1]
        ent = self._plan_for(M, h, w, x.device, nw)
        s = self.upscale_factor
        out = torch.empty((nw * M, 3, s * h, s * w), dtype=torch.float32, device=x.device)
        _lib.check(_lib.lib().vsr_srfbn_debug_premix(ent["plan"], out.data_ptr(),
                                                     torch.cuda.current_stream().cuda_stream), "srfbn_debug_premix")
        return out

    def profile(self, enable=True):
        """Bracket every kernel launch of subsequent forwards with CUDA events (bench.py)."""
        for ent in self._plans.values():
            _lib.check(_lib.lib().vsr_srfbn_profile_enable(ent["plan"], int(bool(enable))), "srfbn_profile_enable")

    def profile_read(self):
        """{kernel class: dict(ms, launches, flops, bytes)} of the last forward of each plan, summed."""
        L = _lib.lib()
        n = 10            # VSR_SRFBN_KERNEL_CLASSES
        out = {}
        for ent in self._plans.values():
            ms = (ctypes.c_double * n)()
            la = (ctypes.c_int32 * n)()
            fl = (ctypes.c_double * n)()
            by = (ctypes.c_double * n)()
            _lib.check(L.vsr_srfbn_profile_read(ent["plan"], ms, la, fl, by), "srfbn_profile_read")
            for k in range(n):
                name = L.vsr_srfbn_kernel_class_name(k).decode()
                d = out.setdefault(name, {"ms": 0.0, "launches": 0, "flops": 0.0, "bytes": 0.0})
                d["ms"] += ms[k]
                d["launches"] += la[k]
                d["flops"] += fl[k]
                d["bytes"] += by[k]
        return out

    def __del__(self):
        try:
            L = _lib.lib()
            for ent in self._plans.values():
                L.vsr_srfbn_plan_destroy(ent["plan"])
        except Exception:
            pass
