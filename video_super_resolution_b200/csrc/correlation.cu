// correlation.cu -- FlowNetC cost volume (SURVEY.md 8f rank 1; not on the warp-and-fuse hot path).
//   ref: correlation_package/correlation_cuda.cc:10-86 (output geometry, zero padding),
//        correlation_cuda_kernel.cu:46-147 (channels_first repack + correlation_forward),
//        correlation.py:7-30; FlowNetC use: pad 20, kernel 1, max_displacement 20, strides 1 / 2
//        (FlowNetC.py:22) -> 441 output channels.
//
//   out[n, (tj+R)*D + (ti+R), y, x] = 1/(k*k*C) * sum_{j,i in kernel} sum_c
//         pad(in1)[n, c, y1+j, x1+i] * pad(in2)[n, c, y1+j + tj*s2, x1+i + ti*s2]
//   y1 = y*s1 + max_displacement (padded coordinates), R = max_displacement / s2, D = 2R+1.
//
// The reference repacks both inputs into zero-padded NHWC copies and then spends one 32-thread block
// per output PIXEL, re-reading the C channels of both images for each of the D*D displacements
// through a warp-shuffle reduction.  Here a warp owns 32 consecutive output x of one (n, y, tj):
// lane = x keeps the D accumulators of its pixel in registers, in1 is read once per channel and the D
// shifted in2 values are coalesced, L1-resident loads; no repack, no padding copy, no reduction.
//
// Arithmetic contract (both forward kernels, restated by oracle.c::or_correlation with padded = 1): one fp32 fmaf
// chain per output over the window taps (j, i) and then the channels c, then __fdiv_rn(acc, k*k*C).  A position
// outside the image reads as zero and its products are taken, as in the reference's zero-padded copies: an Inf or NaN
// that meets padding makes NaN.  (The reference sums 32 strided partials and tree-reduces them, so it agrees to fp32
// rounding, not bit for bit.)
#include "common.cuh"

#include <stdlib.h>

namespace vsr {
namespace {

constexpr int kThreads = 256;
constexpr int kMaxD = 21;   // displacements per axis kept in registers (FlowNetC: 21)

__global__ void __launch_bounds__(kThreads)
correlation_forward_kernel(const float* __restrict__ in1, const float* __restrict__ in2, float* __restrict__ out,
                           int B, int C, int H, int W, int outH, int outW, int pad, int ksize, int maxdisp, int s1, int s2,
                           int R, int D, int segs) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = ((int64_t)blockIdx.x * kThreads + threadIdx.x) >> 5;
  const int64_t n_tasks = (int64_t)B * outH * D * segs;
  const int64_t n_warps = ((int64_t)gridDim.x * kThreads) >> 5;
  const int krad = (ksize - 1) / 2;
  const int64_t HW = (int64_t)H * W;
  for (int64_t task = warp_global; task < n_tasks; task += n_warps) {
    const int seg = (int)(task % segs);
    int64_t r = task / segs;
    const int tjw = (int)(r % D);      // tj + R
    r /= D;
    const int y = (int)(r % outH);
    const int n = (int)(r / outH);
    const int x = seg * 32 + lane;
    // unpadded coordinates of the two window centres
    const int ya = y * s1 + maxdisp - pad, xa = x * s1 + maxdisp - pad;
    const int yb = ya + (tjw - R) * s2;
    float acc[kMaxD];
#pragma unroll
    for (int t = 0; t < kMaxD; ++t) acc[t] = 0.0f;
    const float* p1 = in1 + (int64_t)n * C * HW;
    const float* p2 = in2 + (int64_t)n * C * HW;
    const bool lane_ok = x < outW;
    for (int j = -krad; j <= krad; ++j) {
      const int y1 = ya + j, y2 = yb + j;
      // a zero-padded row still takes its products: 0 * Inf on the other side is NaN, as in the reference
      const bool row1 = lane_ok && (y1 >= 0) && (y1 < H), row2 = lane_ok && (y2 >= 0) && (y2 < H);
      for (int i = -krad; i <= krad; ++i) {
        const int x1 = xa + i;
        const bool in_a = row1 && (x1 >= 0) && (x1 < W);
        const float* a_ptr = p1 + (in_a ? (int64_t)y1 * W + x1 : 0);
        const float* b_row = p2 + (row2 ? (int64_t)y2 * W : 0);
        for (int c = 0; c < C; ++c) {
          const float a = in_a ? __ldg(a_ptr + (int64_t)c * HW) : 0.0f;
          const float* b_c = b_row + (int64_t)c * HW;
#pragma unroll
          for (int t = 0; t < kMaxD; ++t) {
            if (t < D) {
              const int x2 = x1 + (t - R) * s2;
              const float b = (row2 && x2 >= 0 && x2 < W) ? __ldg(b_c + x2) : 0.0f;
              acc[t] = fmaf(a, b, acc[t]);
            }
          }
        }
      }
    }
    if (x < outW) {
      const float nelems = (float)(ksize * ksize * C);
      float* o = out + (((int64_t)n * D * D + (int64_t)tjw * D) * outH + y) * outW + x;
#pragma unroll
      for (int t = 0; t < kMaxD; ++t)
        if (t < D) o[(int64_t)t * outH * outW] = __fdiv_rn(acc[t], nelems);
    }
  }
}


// ---------------------------------------------------------------------------------------------------------
// Fast path for FlowNetC's configuration (kernel_size 1, stride1 1, stride2 2; FlowNetC.py:22): the cost volume of
// one (n, y, tj) row pair is a banded product out[x, ti] = sum_c A[c, x] * B[c, x + 2*(ti-R)] -- register-tiled.
// A warp owns 128 consecutive x of one row pair.  Channels are staged 8 at a time in shared memory with the two
// row segments DE-INTERLEAVED BY COLUMN PARITY, because every displacement is even: a thread that owns the four
// same-parity columns x, x+2, x+4, x+6 then needs 4 contiguous A values and 24 contiguous B values per channel --
// 7 16-byte shared loads for 84 FMAs, against one global load per FMA in the generic kernel above (which was
// L1-bound at 2 TFLOP/s).  Same fp32 FMA chain in channel order and the same padding rule as the generic kernel:
// identical bits, non-finite inputs included.
// Padding follows the reference: a padded row is staged as zeros and its products are taken (0 * Inf is NaN).  A task
// whose in2 row is padding and in1 row is not (about 8 % of FlowNetC's) would run the chain fmaf(a, 0, acc) over the
// channels, the same for every displacement ti of its row: +0, or NaN where a column of in1 holds an Inf or NaN.  The
// zero-displacement task of the same (n, y, x-tile) reads that in1 row anyway; it runs this chain beside its own (one
// fmaf per staged value) and writes those tasks' outputs, which are skipped.
// ---------------------------------------------------------------------------------------------------------
constexpr int kCorrCc = 8;                     // channels per staging round
constexpr int kCorrXT = 128;                   // output columns per warp task
constexpr int kCorrWarps = 4;
constexpr int kCorrBW = kCorrXT + 2 * (kMaxD - 1);   // 168 columns of the second image per task

__global__ void __launch_bounds__(32 * kCorrWarps)
correlation_s2_kernel(const float* __restrict__ in1, const float* __restrict__ in2, float* __restrict__ out, int B,
                      int C, int H, int W, int outH, int outW, int off, int R, int D, int xtiles) {
  __shared__ __align__(16) float sA[kCorrWarps][kCorrCc][2][kCorrXT / 2];
  __shared__ __align__(16) float sB[kCorrWarps][kCorrCc][2][kCorrBW / 2];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int par = lane >> 4, q = lane & 15;    // a quarter-warp shares the parity: conflict-free 16-byte loads
  const int64_t warp_global = (int64_t)blockIdx.x * kCorrWarps + wib;
  const int64_t n_warps = (int64_t)gridDim.x * kCorrWarps;
  const int64_t n_tasks = (int64_t)B * outH * D * xtiles;
  const int64_t HW = (int64_t)H * W;
  float (*A)[2][kCorrXT / 2] = sA[wib];
  float (*Bs)[2][kCorrBW / 2] = sB[wib];
  for (int64_t task = warp_global; task < n_tasks; task += n_warps) {
    const int xt = (int)(task % xtiles);
    int64_t r = task / xtiles;
    const int tjw = (int)(r % D);
    r /= D;
    const int y = (int)(r % outH);
    const int n = (int)(r / outH);
    const int x0 = xt * kCorrXT;
    const int ya = y + off, yb = ya + (tjw - R) * 2;
    const int xs = x0 + off;                      // in1 column of output column x0
    const bool row_a = ya >= 0 && ya < H, row_b = yb >= 0 && yb < H;
    if (row_a && !row_b) continue;                // written by the task with tjw == R (below)
    float acc[4][kMaxD];
    float chk[kCorrXT / 32] = {};                 // slot j: fmaf(a, 0, .) over the channels
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int t = 0; t < kMaxD; ++t) acc[k][t] = 0.0f;
    const float* p1 = in1 + (int64_t)n * C * HW + (int64_t)(row_a ? ya : 0) * W;
    const float* p2 = in2 + (int64_t)n * C * HW + (int64_t)(row_b ? yb : 0) * W;
    // validity of this lane's staging slots, once per task (bit j: slot lane + 32 j); a padded row stages zeros
    uint32_t okA = 0, okB = 0;
#pragma unroll
    for (int j = 0; j < kCorrXT / 32; ++j) {
      const int xi = lane + 32 * j, gx = xs + xi;
      okA |= (uint32_t)(row_a && gx >= 0 && gx < W && x0 + xi < outW) << j;
    }
#pragma unroll
    for (int j = 0; j < (kCorrBW + 31) / 32; ++j) {
      const int xi = lane + 32 * j, gx = xs - 2 * R + xi;
      okB |= (uint32_t)(row_b && xi < kCorrBW && gx >= 0 && gx < W) << j;
    }
    const float* q1 = p1 + xs + lane;
    const float* q2 = p2 + xs - 2 * R + lane;
    float* dA = &A[0][lane & 1][lane >> 1];            // slot lane + 32 j -> [(lane&1)][(lane>>1) + 16 j]
    float* dB = &Bs[0][lane & 1][lane >> 1];
    for (int c0 = 0; c0 < C; c0 += kCorrCc) {
      const int nc = min(kCorrCc, C - c0);
#pragma unroll
      for (int c = 0; c < kCorrCc; ++c) {
        const uint32_t mA = c < nc ? okA : 0u, mB = c < nc ? okB : 0u;
        const float* r1 = q1 + (int64_t)(c0 + c) * HW;
        const float* r2 = q2 + (int64_t)(c0 + c) * HW;
#pragma unroll
        for (int j = 0; j < kCorrXT / 32; ++j) {
          const float v = ((mA >> j) & 1u) ? __ldg(r1 + 32 * j) : 0.0f;
          dA[c * kCorrXT + 16 * j] = v;
          chk[j] = fmaf(v, 0.0f, chk[j]);
        }
#pragma unroll
        for (int j = 0; j < (kCorrBW + 31) / 32; ++j)
          if (lane + 32 * j < kCorrBW) dB[c * kCorrBW + 16 * j] = ((mB >> j) & 1u) ? __ldg(r2 + 32 * j) : 0.0f;
      }
      __syncwarp();
#pragma unroll 2
      for (int c = 0; c < kCorrCc; ++c) {
        const float4 a4 = *reinterpret_cast<const float4*>(&A[c][par][4 * q]);
        const float a[4] = {a4.x, a4.y, a4.z, a4.w};
        float bb[24];
#pragma unroll
        for (int j = 0; j < 6; ++j) {
          const float4 b4 = *reinterpret_cast<const float4*>(&Bs[c][par][4 * q + 4 * j]);
          bb[4 * j] = b4.x; bb[4 * j + 1] = b4.y; bb[4 * j + 2] = b4.z; bb[4 * j + 3] = b4.w;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
          for (int t = 0; t < kMaxD; ++t)
            if (t < D) acc[k][t] = fmaf(a[k], bb[k + t], acc[k][t]);
      }
      __syncwarp();
    }
    // transpose through shared memory so that the stores are 128 contiguous floats per displacement
    const float nelems = (float)C;
    float* S = &A[0][0][0];
    float* o = out + (((int64_t)n * D * D + (int64_t)tjw * D) * outH + y) * outW + x0;
#pragma unroll
    for (int t = 0; t < kMaxD; ++t) {
      if (t < D) {
#pragma unroll
        for (int k = 0; k < 4; ++k) S[8 * q + par + 2 * k] = __fdiv_rn(acc[k][t], nelems);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < kCorrXT / 32; ++j) {
          const int xi = lane + 32 * j;
          if (x0 + xi < outW) o[(int64_t)t * outH * outW + xi] = S[xi];
        }
        __syncwarp();
      }
    }
    if (tjw == R && row_a) {                      // the skipped tasks of this in1 row whose in2 row is padding
      float z[kCorrXT / 32];
#pragma unroll
      for (int j = 0; j < kCorrXT / 32; ++j) z[j] = __fdiv_rn(chk[j], nelems);   // column lane + 32 j
      for (int tp = 0; tp < D; ++tp) {
        const int yp = ya + (tp - R) * 2;
        if (yp >= 0 && yp < H) continue;
        float* op = out + (((int64_t)n * D * D + (int64_t)tp * D) * outH + y) * outW + x0;
        for (int t = 0; t < D; ++t)
#pragma unroll
          for (int j = 0; j < kCorrXT / 32; ++j) {
            const int xi = lane + 32 * j;
            if (x0 + xi < outW) op[(int64_t)t * outH * outW + xi] = z[j];
          }
      }
    }
  }
}


// ---------------------------------------------------------------------------------------------------------
// Backward (completes the CorrelationFunction surface; correlation_cuda_kernel.cu:148-333, stride1 = 1 -- for
// stride1 > 1 the reference writes gradInput out of bounds).  One thread per input element (n, c, Y, X), X fastest:
//   gradInput1[n,c,Y,X] = 1/(k*k*C) * sum_tc in2[n,c,Y + j2, X + i2] * sum_window gradOutput[n,tc,.,.]
//   gradInput2[n,c,Y,X] = 1/(k*k*C) * sum_tc in1[n,c,Y - j2, X - i2] * sum_{window shifted by (j2,i2)} gradOutput[n,tc,.,.]
// the window being the outputs whose kernel footprint covers the pixel (one output for kernel_size 1).  Both the
// gradOutput and the shifted-image loads are coalesced along X.  One fp32 fmaf chain per element over tj, ti and the
// clamped window rows j and columns i, then __fdiv_rn(acc, k*k*C) (restated by
// oracle.c::or_correlation_backward_chain).  The other image is zero outside itself and those products are taken, so
// an Inf or NaN of gradOutput that meets padding makes NaN, as in the reference (which sums 32 strided partials and
// reduces them: equal to fp32 rounding, not bit for bit).
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
correlation_backward_kernel(const float* __restrict__ other, const float* __restrict__ gout, float* __restrict__ gin,
                            int which, int B, int C, int H, int W, int outH, int outW, int pad, int ksize, int maxdisp,
                            int s2, int R, int D) {
  const int64_t HW = (int64_t)H * W, OHW = (int64_t)outH * outW;
  const int64_t total = (int64_t)B * C * HW;
  const int krad = (ksize - 1) / 2;
  const float nelems = (float)(ksize * ksize * C);
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int X = (int)(idx % W);
    const int Y = (int)((idx / W) % H);
    const int64_t nc = idx / HW;
    const int n = (int)(nc / C);
    const int y = Y + pad, x = X + pad;
    const float* img = other + nc * HW;
    const float* g = gout + (int64_t)n * D * D * OHW;
    float acc = 0.0f;
    for (int tj = 0; tj < D; ++tj) {
      const int j2 = (tj - R) * s2;
      const int oy = (which ? y - j2 : y + j2) - pad;
      const bool row_in = oy >= 0 && oy < H;                 // else the other image's row is zero padding
      int ymin = y - krad - maxdisp - (which ? j2 : 0), ymax = ymin + 2 * krad;
      if (ymax < 0 || ymin >= outH) continue;
      ymin = max(ymin, 0);
      ymax = min(ymax, outH - 1);
      for (int ti = 0; ti < D; ++ti) {
        const int i2 = (ti - R) * s2;
        const int ox = (which ? x - i2 : x + i2) - pad;
        int xmin = x - krad - maxdisp - (which ? i2 : 0), xmax = xmin + 2 * krad;
        if (xmax < 0 || xmin >= outW) continue;
        xmin = max(xmin, 0);
        xmax = min(xmax, outW - 1);
        const float val = (row_in && ox >= 0 && ox < W) ? __ldg(img + (int64_t)oy * W + ox) : 0.0f;
        const float* gt = g + (int64_t)(tj * D + ti) * OHW;
        for (int j = ymin; j <= ymax; ++j)
          for (int i = xmin; i <= xmax; ++i) acc = fmaf(__ldg(gt + (int64_t)j * outW + i), val, acc);
      }
    }
    gin[idx] = __fdiv_rn(acc, nelems);
  }
}

}  // namespace
}  // namespace vsr

using namespace vsr;

extern "C" int vsr_correlation_output_shape(int C, int H, int W, int pad_size, int kernel_size, int max_displacement,
                                            int stride1, int stride2, int* out_channels, int* out_h, int* out_w) {
  (void)C;
  if (H <= 0 || W <= 0 || pad_size < 0 || kernel_size < 1 || (kernel_size & 1) == 0 || max_displacement < 0 || stride1 < 1 ||
      stride2 < 1 || !out_channels || !out_h || !out_w)
    return VSR_ERR_INVALID_ARG;
  // correlation_cuda.cc:25-34
  const int border = (kernel_size - 1) / 2 + max_displacement;
  const int ph = H + 2 * pad_size, pw = W + 2 * pad_size;
  const int D = (max_displacement / stride2) * 2 + 1;
  *out_channels = D * D;
  *out_h = (ph - 2 * border + stride1 - 1) / stride1;
  *out_w = (pw - 2 * border + stride1 - 1) / stride1;
  if (*out_h <= 0 || *out_w <= 0) return VSR_ERR_UNSUPPORTED;
  return VSR_OK;
}

extern "C" int vsr_correlation_forward(const float* input1, const float* input2, float* output, int B, int C, int H, int W,
                                       int pad_size, int kernel_size, int max_displacement, int stride1, int stride2,
                                       int corr_multiply, vsr_stream_t stream) {
  (void)corr_multiply;   // accepted and unused, as in correlation_cuda_kernel.cu:73-147
  if (!input1 || !input2 || !output || B <= 0 || C <= 0) return VSR_ERR_INVALID_ARG;
  int oc, oh, ow;
  int rc = vsr_correlation_output_shape(C, H, W, pad_size, kernel_size, max_displacement, stride1, stride2, &oc, &oh, &ow);
  if (rc) return rc;
  const int R = max_displacement / stride2, D = 2 * R + 1;
  if (D > kMaxD) return VSR_ERR_UNSUPPORTED;
  if (kernel_size == 1 && stride1 == 1 && stride2 == 2 && !getenv("VSR_CORR_GENERIC")) {   // FlowNetC's configuration
    const int xtiles = ceil_div(ow, kCorrXT);
    const int64_t tasks = (int64_t)B * oh * D * xtiles;
    int64_t blocks = ceil_div64(tasks, kCorrWarps);
    const int64_t cap = (int64_t)kNumSMs * 64;
    if (blocks > cap) blocks = cap;
    correlation_s2_kernel<<<(int)blocks, 32 * kCorrWarps, 0, as_stream(stream)>>>(
        input1, input2, output, B, C, H, W, oh, ow, max_displacement - pad_size, R, D, xtiles);
    return after_launch();
  }
  const int segs = ceil_div(ow, 32);
  const int64_t n_tasks = (int64_t)B * oh * D * segs;
  int64_t blocks = ceil_div64(n_tasks, kThreads / 32);
  const int64_t cap = (int64_t)kNumSMs * 8 * 8;
  if (blocks > cap) blocks = cap;
  correlation_forward_kernel<<<(int)blocks, kThreads, 0, as_stream(stream)>>>(input1, input2, output, B, C, H, W, oh, ow,
                                                                             pad_size, kernel_size, max_displacement,
                                                                             stride1, stride2, R, D, segs);
  return after_launch();
}

extern "C" int vsr_correlation_backward(const float* input1, const float* input2, const float* grad_output,
                                        float* grad_input1, float* grad_input2, int B, int C, int H, int W, int pad_size,
                                        int kernel_size, int max_displacement, int stride1, int stride2, int corr_multiply,
                                        vsr_stream_t stream) {
  (void)corr_multiply;
  if (!input1 || !input2 || !grad_output || !grad_input1 || !grad_input2 || B <= 0 || C <= 0) return VSR_ERR_INVALID_ARG;
  if (stride1 != 1) return VSR_ERR_UNSUPPORTED;   // the reference's backward indexes out of bounds for stride1 > 1
  int oc, oh, ow;
  int rc = vsr_correlation_output_shape(C, H, W, pad_size, kernel_size, max_displacement, stride1, stride2, &oc, &oh, &ow);
  if (rc) return rc;
  const int R = max_displacement / stride2, D = 2 * R + 1;
  const int64_t total = (int64_t)B * C * H * W;
  int64_t blocks = ceil_div64(total, kThreads);
  const int64_t cap = (int64_t)kNumSMs * 8 * 8;
  if (blocks > cap) blocks = cap;
  cudaStream_t st = as_stream(stream);
  correlation_backward_kernel<<<(int)blocks, kThreads, 0, st>>>(input2, grad_output, grad_input1, 0, B, C, H, W, oh, ow,
                                                               pad_size, kernel_size, max_displacement, stride2, R, D);
  rc = after_launch();
  if (rc) return rc;
  correlation_backward_kernel<<<(int)blocks, kThreads, 0, st>>>(input1, grad_output, grad_input2, 1, B, C, H, W, oh, ow,
                                                               pad_size, kernel_size, max_displacement, stride2, R, D);
  return after_launch();
}
