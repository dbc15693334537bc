// stack.cu -- assembly of the (M,3,h,w) map stack the fusion convolutions consume (a7), and the
// estimate slot of the second (fuse) pass.
//   ref: network/video_super_resolution.py:33-40 (torch.cat of frames, flow maps, depth maps tiled x3 by
//        maskprocess, estimate; NHWC->NCHW via transpose1323), :43-44 / :57-62 (nearest downsize of the
//        first-pass output, MaskedArray fill with the VOS mask, second torch.cat).
// The reference builds the stack with 6 transposes, 3 interpolates and 2 cats (each a full pass over
// memory, some through numpy on the host); here it is one pass: every input is read once and every
// output plane is written once with coalesced stores.
#include "common.cuh"

namespace vsr {
namespace {

constexpr int kThreads = 256;

// Stack order (video_super_resolution.py:40, generalised to T frames, SURVEY.md Appendix D):
//   maps [0,T)        frames: warped neighbours with the centre frame in its place
//   maps [T,2T-1)     flow maps: (projected fx, projected fy, warp-residual norm)
//   maps [2T-1,3T-2)  depth maps: one channel tiled x3 (utils/tools.py:76-77)
//   map  3T-2         estimate (written by estimate_slot_kernel or copied from `estimate`)
__global__ void __launch_bounds__(kThreads)
assemble_stack_kernel(const float* __restrict__ warped,   // (T-1,h,w,3) NHWC
                      const float* __restrict__ centre,   // (h,w,3)
                      const float* __restrict__ proj,     // (T-1,h,w,2)
                      const float* __restrict__ resid,    // (T-1,h,w)
                      const float* __restrict__ depth,    // (T-1,h,w)
                      const float* __restrict__ estimate, // (3,h,w) NCHW or nullptr (-> fallback frame)
                      const float* __restrict__ fallback, // (h,w,3) NHWC: LR frame 0 of the window
                                                          // (video_super_resolution.py:37-38 `data_clone[0:1]`)
                      float* __restrict__ stack, int T, int centre_idx, int64_t hw, int64_t frame_stride) {
  // blockIdx.y: the frame window.  Per window: warped / proj / resid / depth advance by their (T-1) images, the stack by
  // its M = 3T-1 maps, the estimate by one (3,h,w) image, centre and fallback by frame_stride floats.
  if (blockIdx.y) {
    const int64_t wb = blockIdx.y;
    warped += wb * (T - 1) * hw * 3;
    proj += wb * (T - 1) * hw * 2;
    resid += wb * (T - 1) * hw;
    depth += wb * (T - 1) * hw;
    stack += wb * (3 * T - 1) * 3 * hw;
    centre += wb * frame_stride;
    if (estimate) estimate += wb * 3 * hw;
    else fallback += wb * frame_stride;
  }
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < hw; p += (int64_t)gridDim.x * blockDim.x) {
    const float c0 = __ldg(centre + p * 3), c1 = __ldg(centre + p * 3 + 1), c2 = __ldg(centre + p * 3 + 2);
    for (int t = 0, n = 0; t < T; ++t) {
      float v0 = c0, v1 = c1, v2 = c2;
      if (t != centre_idx) {
        const float* s = warped + ((int64_t)n * hw + p) * 3;
        v0 = __ldg(s); v1 = __ldg(s + 1); v2 = __ldg(s + 2);
        ++n;
      }
      float* o = stack + (int64_t)t * 3 * hw + p;
      o[0] = v0; o[hw] = v1; o[2 * hw] = v2;
    }
    for (int n = 0; n < T - 1; ++n) {
      const float2 f = __ldg(reinterpret_cast<const float2*>(proj) + (int64_t)n * hw + p);
      float* o = stack + (int64_t)(T + n) * 3 * hw + p;
      o[0] = f.x; o[hw] = f.y; o[2 * hw] = __ldg(resid + (int64_t)n * hw + p);
      const float d = __ldg(depth + (int64_t)n * hw + p);
      float* od = stack + (int64_t)(2 * T - 1 + n) * 3 * hw + p;
      od[0] = d; od[hw] = d; od[2 * hw] = d;
    }
    float* oe = stack + (int64_t)(3 * T - 2) * 3 * hw + p;
    if (estimate) { oe[0] = __ldg(estimate + p); oe[hw] = __ldg(estimate + hw + p); oe[2 * hw] = __ldg(estimate + 2 * hw + p); }
    else { oe[0] = __ldg(fallback + p * 3); oe[hw] = __ldg(fallback + p * 3 + 1); oe[2 * hw] = __ldg(fallback + p * 3 + 2); }
  }
}

// slot[c,y,x] = mask[y,x] ? 0 : hr[c, y*s, x*s]: F.interpolate(..., size) default 'nearest' picks
// floor(dst * in/out) = dst*s (video_super_resolution.py:44), then MaskedArray(...).filled(0) (:58-60).
__global__ void __launch_bounds__(kThreads)
estimate_slot_kernel(const float* __restrict__ hr, const uint8_t* __restrict__ mask, float* __restrict__ slot, int h,
                     int w, int s, int64_t slot_stride) {
  const int64_t hw = (int64_t)h * w, HW = hw * s * s;
  if (blockIdx.y) {     // window blockIdx.y: hr (3,H,W) and mask (h,w) images in sequence, slots slot_stride floats apart
    const int64_t wb = blockIdx.y;
    hr += wb * 3 * HW;
    if (mask) mask += wb * hw;
    slot += wb * slot_stride;
  }
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < hw; p += (int64_t)gridDim.x * blockDim.x) {
    const int y = (int)(p / w), x = (int)(p - (int64_t)y * w);
    const bool m = mask != nullptr && __ldg(mask + p) != 0;
    const int64_t q = (int64_t)y * s * (w * s) + (int64_t)x * s;
#pragma unroll
    for (int c = 0; c < 3; ++c) slot[c * hw + p] = m ? 0.0f : __ldg(hr + c * HW + q);
  }
}

inline int grid_for(int64_t n) {
  int64_t b = ceil_div64(n, kThreads), cap = (int64_t)kNumSMs * 8;
  return (int)(b > cap ? cap : (b < 1 ? 1 : b));
}

}  // namespace
}  // namespace vsr

using namespace vsr;

extern "C" int vsr_assemble_stack_windows(const float* warped, const float* centre, const float* proj,
                                          const float* resid, const float* depth, const float* estimate,
                                          const float* fallback, float* stack, int windows, int64_t frame_stride, int T,
                                          int centre_idx, int h, int w, vsr_stream_t stream) {
  if (!warped || !centre || !proj || !resid || !depth || !stack || windows < 1 || windows > 65535 || frame_stride < 0 ||
      T < 2 || centre_idx < 0 || centre_idx >= T || h <= 0 || w <= 0 || (!estimate && !fallback))
    return VSR_ERR_INVALID_ARG;
  if (reinterpret_cast<uintptr_t>(proj) % 8) return VSR_ERR_INVALID_ARG;
  const int64_t hw = (int64_t)h * w;
  assemble_stack_kernel<<<dim3(grid_for(hw), windows), kThreads, 0, as_stream(stream)>>>(
      warped, centre, proj, resid, depth, estimate, fallback, stack, T, centre_idx, hw, frame_stride);
  return after_launch();
}

extern "C" int vsr_estimate_slot_windows(const float* hr, const uint8_t* mask, float* slot, int windows,
                                         int64_t slot_stride, int h, int w, int scale, vsr_stream_t stream) {
  if (!hr || !slot || windows < 1 || windows > 65535 || slot_stride < 0 || h <= 0 || w <= 0 || scale < 1)
    return VSR_ERR_INVALID_ARG;
  estimate_slot_kernel<<<dim3(grid_for((int64_t)h * w), windows), kThreads, 0, as_stream(stream)>>>(hr, mask, slot, h, w,
                                                                                                   scale, slot_stride);
  return after_launch();
}
