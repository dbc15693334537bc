"""VSR -- the pipeline model with the reference's call sites (network/video_super_resolution.py:12-69).

    VSR(window=3, flow_estimator=None, depth_estimator=None, vos_estimator=None)
    .forward(data (T,h,w,3), target, high_frames (T,H,W,3), estimated_image (1,H,W,3)|None, train=False)
        -> (output (1,H,W,3), loss|None)

Same module attributes (`model`, `FlowModule`, `DepthModule`, `VOSModule`), same tensor layouts (NHWC
0..255 fp32 in and out, Appendix D of SURVEY.md), same two-pass structure: pass 1 builds the map
stack and runs the fusion convs (:24-41), pass 2 replaces the estimate slot by the downsized,
VOS-masked first-pass output and runs them again (:43-64).  Differences, all forced by scope:
  * the learned estimators are pluggable callables (the reference hard-loads absent pretrained
    weights); `forward_geometry` takes flow / inverse depth / logits directly, which is what the
    benchmarks and tests use;
  * the window is T frames (the reference hard-wires 3), M = 3T-1 maps;
  * losses (loss_function.py) are out of scope: `train=True` raises.
`map_group=pg` (an NCCL process group) runs every window over the group's GPUs (pipeline.WarpFusePipeline,
DESIGN.md 11); every rank of the group calls forward with the same inputs and gets the same frame.
"""
import torch

from ..my_packages.DepthProjection.DepthProjectionModule import DepthProjectionModule
from ..my_packages.FlowProjection.FlowProjectionModule import FlowProjectionModule
from ..my_packages.SRProjection.SRProjectionModule import SRProjectionModule
from ..my_packages.VOSProjection.VOSProjectionModule import VOSProjectionModule
from ..pipeline import WarpFusePipeline
from ..utils.tools import transpose1312


class VSR(torch.nn.Module):
    def __init__(self, window=3, flow_estimator=None, depth_estimator=None, vos_estimator=None, map_group=None):
        super(VSR, self).__init__()
        self.window = window
        self.model = SRProjectionModule(num_maps=3 * window - 1, map_group=map_group)
        self.FlowModule = FlowProjectionModule(estimator=flow_estimator).eval()
        self.DepthModule = DepthProjectionModule(estimator=depth_estimator).eval()
        self.VOSModule = VOSProjectionModule(estimator=vos_estimator).eval()
        self._pipes = {}

    def _pipe(self, h, w, device, windows=1):
        key = (h, w, device.index) + ((windows,) if windows > 1 else ())
        if key not in self._pipes:
            self._pipes[key] = WarpFusePipeline(self.window, h, w, self.model, self.model.upscale_factor, device=device,
                                                windows=windows, map_group=self.model.map_group)
        return self._pipes[key]

    def forward_geometry(self, data, flows, inv_depth, logits_a, logits_b, estimated_image=None):
        """data (T,h,w,3); flows (T-1,h,w,2); inv_depth (T-1,h,w); logits (h,w) x2; estimated_image
        (1,H,W,3)|None -> output (1,H,W,3)."""
        T, h, w, _ = data.shape
        pipe = self._pipe(h, w, data.device)
        est = None
        if estimated_image is not None:
            # interpolate(transpose1323(estimated_image), data_shape): nearest = every s-th pixel (:37)
            s = self.model.upscale_factor
            est = estimated_image[0].permute(2, 0, 1)[:, ::s, ::s].contiguous()
        with torch.no_grad():
            out = pipe.step(data.contiguous(), flows.contiguous(), inv_depth.contiguous(), logits_a.contiguous(),
                            logits_b.contiguous(), est)
        return transpose1312(out)                                   # (1,3,H,W) -> (1,H,W,3), :64

    def forward(self, data, target, high_frames, estimated_image, train=False):
        if train:
            raise NotImplementedError("losses (loss_function.py) are outside the B200 hot path")
        T = data.shape[0]
        c = T // 2
        if self.FlowModule.estimator is None or self.DepthModule.estimator is None or self.VOSModule.estimator is None:
            raise RuntimeError("VSR.forward needs flow / depth / segmentation estimators (out of scope here); "
                               "attach callables or use forward_geometry(...)")
        flows = torch.stack([self.FlowModule.estimator(data[t], data[t + 1]) for t in range(T - 1)])
        inv_depth = torch.stack([self.DepthModule.estimator(data[t:t + 2])[1] for t in range(T - 1)])
        la, lb = self.VOSModule.estimator(data[max(c - 1, 0)], data[c])
        output = self.forward_geometry(data, flows, inv_depth, la, lb, estimated_image)
        if high_frames is not None:
            high_frames[min(1, high_frames.shape[0] - 1)] = output[0]   # :66
        return output, None
