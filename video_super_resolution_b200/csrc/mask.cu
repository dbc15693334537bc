// mask.cu -- the elementwise integer part of VOSProjection (a5): threshold of the two sigmoid
// side outputs and the mask fill of the estimate.
//   ref: my_packages/VOSProjection/VOSProjectionModule.py:22-25
//        network/video_super_resolution.py:58-60, utils/tools.py:76-77
// The reference does both on the host through numpy (three device<->host round trips per frame);
// here they are two trivially bandwidth-bound kernels on the caller's stream.
#include "common.cuh"

namespace vsr {
namespace {

constexpr int kThreads = 256;

// sigmoid in double, rounded to fp32; fp32 sum; fp32 compare against (float)0.7 -- the same
// sequence as oracle.c::or_vos_threshold, so the {0,1} mask is bit-exact.
__global__ void __launch_bounds__(kThreads)
vos_threshold_kernel(const float* __restrict__ la, const float* __restrict__ lb, uint8_t* __restrict__ mask, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float sa = __double2float_rn(__ddiv_rn(1.0, __dadd_rn(1.0, exp(-(double)__ldg(la + i)))));
    float sb = __double2float_rn(__ddiv_rn(1.0, __dadd_rn(1.0, exp(-(double)__ldg(lb + i)))));
    float s = __fadd_rn(sa, sb);
    mask[i] = s > 0.7f ? 1 : 0;
  }
}

__global__ void __launch_bounds__(kThreads)
mask_fill_kernel(const float* __restrict__ image, const uint8_t* __restrict__ mask, float* __restrict__ out, int C,
                 int64_t hw) {
  const int64_t n = (int64_t)C * hw;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t p = i % hw;
    out[i] = __ldg(mask + p) ? 0.0f : __ldg(image + i);
  }
}

inline int grid_for(int64_t n) {
  int64_t blocks = ceil_div64(n, kThreads);
  int64_t cap = (int64_t)kNumSMs * 8 * 4;
  return (int)(blocks > cap ? cap : (blocks < 1 ? 1 : blocks));
}

}  // namespace
}  // namespace vsr

using namespace vsr;

// windows (h,w) logit pairs in sequence: the threshold is elementwise, so the windows are one flat launch
extern "C" int vsr_vos_threshold_windows(const float* logits_a, const float* logits_b, uint8_t* mask, int windows, int h,
                                         int w, vsr_stream_t stream) {
  if (!logits_a || !logits_b || !mask || windows < 1 || h <= 0 || w <= 0) return VSR_ERR_INVALID_ARG;
  int64_t n = (int64_t)windows * h * w;
  vos_threshold_kernel<<<grid_for(n), kThreads, 0, as_stream(stream)>>>(logits_a, logits_b, mask, n);
  return after_launch();
}

extern "C" int vsr_mask_fill(const float* image, const uint8_t* mask, float* masked, int C, int h, int w,
                             vsr_stream_t stream) {
  if (!image || !mask || !masked || C <= 0 || h <= 0 || w <= 0) return VSR_ERR_INVALID_ARG;
  int64_t hw = (int64_t)h * w;
  mask_fill_kernel<<<grid_for(C * hw), kThreads, 0, as_stream(stream)>>>(image, mask, masked, C, hw);
  return after_launch();
}
