// warp.cu -- backward warps of the hot path: bilinear / nearest resampling by a pixel-unit flow,
// the fused warp-residual channel norm, the u8 label warp and the stand-alone channel norm.
//
// Arithmetic contract (bit for bit, so the result equals the reference kernel's output):
//   ref: my_packages/FlowProjection/networks/resample2d_package/resample2d_kernel.cu:15-72
//        my_packages/FlowProjection/networks/channelnorm_package/channelnorm_kernel.cu:19-60
// What is different is everything around the arithmetic: the flow is read once per pixel instead
// of once per (pixel, channel); tap indices and weights are computed once per pixel; the
// channels-last kernels move 16-byte vectors and stage the C=3 output through shared memory so
// that every global store is a full 128-bit coalesced transaction.
#include <cuda_fp16.h>

#include "common.cuh"

namespace vsr {
namespace {

constexpr int kThreads = 256;

struct Taps {
  int xL, xR, yT, yB;
  double wTL, wTR, wBL;
  float wBR;
  float af, bf;   // alpha, beta in fp32 (fast mode)
};

// `bilinear` argument of the channels-last entry points
constexpr int kModeNearest = 0, kModeExact = 1, kModeFast = 2;

// floor() and float->int without the conversion (XU) pipe, which ncu showed to be the busiest pipe of
// these kernels (55-77 %): for |v| < 2^22 adding and subtracting 1.5*2^23 rounds to an integer on the
// FMA pipe, one compare fixes round-to-nearest into floor, and the integer is read off the mantissa.
// Exact, so the bit-for-bit contract holds; larger magnitudes / NaN take the conversion instructions.
__device__ __forceinline__ float floor_small(float v, bool& ok) {
  ok = fabsf(v) < 4194304.0f;
  const float r = __fsub_rn(__fadd_rn(v, 12582912.0f), 12582912.0f);
  return r > v ? __fsub_rn(r, 1.0f) : r;
}
__device__ __forceinline__ int int_of_small(float r) {   // r integral, |r| <= 2^22
  return __float_as_int(__fadd_rn(r, 12582912.0f)) - 0x4B400000;
}

// resample2d_kernel.cu:40-52: fp32 coordinates, floor, border clamp with the output dims;
// :56-58: the `1.` literals make the TL/TR/BL weights (and products) doubles; :59 the BR term
// `(alpha)*(beta) * in` has no literal, so it is fp32 and nvcc contracts `val += ...` into an FMA
// (verified in the SASS of the reference compiled for sm_100a: FMUL alpha*beta, FFMA).
template <bool FAST = false>
__device__ __forceinline__ Taps bilinear_taps(int x, int y, float dx, float dy, int W, int H) {
  Taps t;
  float xf = __fadd_rn((float)x, dx);
  float yf = __fadd_rn((float)y, dy);
  bool okx, oky;
  float fx0 = floor_small(xf, okx), fy0 = floor_small(yf, oky);
  if (okx && oky) {
    const int ix = int_of_small(fx0), iy = int_of_small(fy0);
    t.xL = max(min(ix, W - 1), 0);
    t.xR = max(min(ix + 1, W - 1), 0);
    t.yT = max(min(iy, H - 1), 0);
    t.yB = max(min(iy + 1, H - 1), 0);
  } else {
    fx0 = floorf(xf);
    fy0 = floorf(yf);
    t.xL = max(min((int)fx0, W - 1), 0);
    t.xR = max(min((int)__fadd_rn(fx0, 1.0f), W - 1), 0);
    t.yT = max(min((int)fy0, H - 1), 0);
    t.yB = max(min((int)__fadd_rn(fy0, 1.0f), H - 1), 0);
  }
  float alpha_f = __fsub_rn(xf, fx0), beta_f = __fsub_rn(yf, fy0);
  t.af = alpha_f;
  t.bf = beta_f;
  if (FAST) return t;
  double alpha = (double)alpha_f, beta = (double)beta_f;
  double ia = __dsub_rn(1.0, alpha), ib = __dsub_rn(1.0, beta);
  t.wTL = __dmul_rn(ia, ib);
  t.wTR = __dmul_rn(alpha, ib);
  t.wBL = __dmul_rn(ia, beta);
  t.wBR = __fmul_rn(alpha_f, beta_f);
  return t;
}

// :56-59 TL,TR,BL: product in double, rounded to fp32, fp32 add; BR: one fp32 FMA
__device__ __forceinline__ float blend_acc(const Taps& t, float v, float tl, float tr, float bl, float br) {
  v = __fadd_rn(v, __double2float_rn(__dmul_rn(t.wTL, (double)tl)));
  v = __fadd_rn(v, __double2float_rn(__dmul_rn(t.wTR, (double)tr)));
  v = __fadd_rn(v, __double2float_rn(__dmul_rn(t.wBL, (double)bl)));
  return fmaf(t.wBR, br, v);
}
__device__ __forceinline__ float blend(const Taps& t, float tl, float tr, float bl, float br) {
  float v = 0.0f;
  v = __fadd_rn(v, __double2float_rn(__dmul_rn(t.wTL, (double)tl)));
  v = __fadd_rn(v, __double2float_rn(__dmul_rn(t.wTR, (double)tr)));
  v = __fadd_rn(v, __double2float_rn(__dmul_rn(t.wBL, (double)bl)));
  v = fmaf(t.wBR, br, v);
  return v;
}

// Fast mode (pipeline default): the same taps and border rule, weights and products in fp32 FMAs.
// Differs from the reference's mixed double/float sequence by a few fp32 ulps (<= 1e-4 on 0..255
// data; the north star allows 1e-3 for warps) and needs no fp64 conversion at all.
__device__ __forceinline__ float blend_fast(const Taps& t, float tl, float tr, float bl, float br) {
  const float ia = 1.0f - t.af, ib = 1.0f - t.bf;
  float top = fmaf(t.af, tr, ia * tl);
  float bot = fmaf(t.af, br, ia * bl);
  return fmaf(t.bf, bot, ib * top);
}
template <bool FAST>
__device__ __forceinline__ float blend_mode(const Taps& t, float tl, float tr, float bl, float br) {
  return FAST ? blend_fast(t, tl, tr, bl, br) : blend(t, tl, tr, bl, br);
}

// :65-70 `floor(xf + 0.5)`: the literal promotes to double; ties go up.  floor(xf + 0.5) evaluated
// exactly equals floor(xf) + (xf - floor(xf) >= 0.5): the subtraction is exact in fp32, so the fp32
// form below returns the reference's integer without touching the fp64 / conversion pipes.
__device__ __forceinline__ void nearest_tap(int x, int y, float dx, float dy, int W, int H, int& xN, int& yN) {
  float xf = __fadd_rn((float)x, dx);
  float yf = __fadd_rn((float)y, dy);
  bool okx, oky;
  const float fx0 = floor_small(xf, okx), fy0 = floor_small(yf, oky);
  if (okx && oky) {
    xN = max(min(int_of_small(fx0) + (__fsub_rn(xf, fx0) >= 0.5f ? 1 : 0), W - 1), 0);
    yN = max(min(int_of_small(fy0) + (__fsub_rn(yf, fy0) >= 0.5f ? 1 : 0), H - 1), 0);
  } else {
    xN = max(min((int)floor(__dadd_rn((double)xf, 0.5)), W - 1), 0);
    yN = max(min((int)floor(__dadd_rn((double)yf, 0.5)), H - 1), 0);
  }
}

// ---------------------------------------------------------------------------------------------
// Reference layout (NCHW).  One thread per (b, y, x); the channel loop re-uses taps and weights.
// Loads/stores are coalesced along x for every channel plane.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
resample2d_nchw_kernel(const float* __restrict__ in1, const float* __restrict__ flow, float* __restrict__ out,
                       int B, int C, int H, int W, int bilinear, const PixDecode pd, int ks) {
  const int64_t HW = (int64_t)H * W;
  const int64_t n = (int64_t)B * HW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int x, y, b;
    decode_pix((uint32_t)i, pd, b, y, x);
    const float* fl = flow + (int64_t)b * 2 * HW + (int64_t)y * W + x;
    float dx = __ldg(fl), dy = __ldg(fl + HW);
    const float* src = in1 + (int64_t)b * C * HW;
    float* dst = out + (int64_t)b * C * HW + (int64_t)y * W + x;
    if (bilinear && ks > 1) {
      // resample2d_kernel.cu:54-61: the four taps are summed again at every offset (fy, fx) of a ks x ks window,
      // un-normalised and UN-CLAMPED: (yT + fy, xL + fx) is plain NCHW address arithmetic, so an offset past the row /
      // plane end reads the next row / plane, exactly as the reference does.  Only addresses past the end of the whole
      // tensor (the reference reads out of bounds there) are pinned to its last element.
      Taps t = bilinear_taps(x, y, dx, dy, W, H);
      const int64_t last = (int64_t)B * C * HW - 1;
      for (int c = 0; c < C; ++c) {
        const int64_t base = ((int64_t)b * C + c) * HW;
        float val = 0.0f;
        for (int fy = 0; fy < ks; ++fy)
          for (int fx = 0; fx < ks; ++fx) {
            const int64_t iTL = base + (int64_t)(t.yT + fy) * W + t.xL + fx, iTR = base + (int64_t)(t.yT + fy) * W + t.xR + fx;
            const int64_t iBL = base + (int64_t)(t.yB + fy) * W + t.xL + fx, iBR = base + (int64_t)(t.yB + fy) * W + t.xR + fx;
            val = blend_acc(t, val, __ldg(in1 + min(iTL, last)), __ldg(in1 + min(iTR, last)), __ldg(in1 + min(iBL, last)),
                            __ldg(in1 + min(iBR, last)));
          }
        dst[(int64_t)c * HW] = val;
      }
    } else if (bilinear) {
      Taps t = bilinear_taps(x, y, dx, dy, W, H);
      int64_t oTL = (int64_t)t.yT * W + t.xL, oTR = (int64_t)t.yT * W + t.xR;
      int64_t oBL = (int64_t)t.yB * W + t.xL, oBR = (int64_t)t.yB * W + t.xR;
#pragma unroll 3
      for (int c = 0; c < C; ++c) {
        const float* p = src + (int64_t)c * HW;
        dst[(int64_t)c * HW] = blend(t, __ldg(p + oTL), __ldg(p + oTR), __ldg(p + oBL), __ldg(p + oBR));
      }
    } else {
      int xN, yN;
      nearest_tap(x, y, dx, dy, W, H, xN, yN);
      int64_t o = (int64_t)yN * W + xN;
      for (int c = 0; c < C; ++c) dst[(int64_t)c * HW] = __ldg(src + (int64_t)c * HW + o);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Channels-last, C == 3 (frames).  A block owns 256 consecutive pixels; results are staged in
// shared memory and leave as 192 coalesced float4 stores.  Optional fused residual norm
// sqrt(sum_c (ref - warped)^2) (models.py:86-88 = resample -> subtract -> channelnorm).
// ---------------------------------------------------------------------------------------------
template <bool FAST>
__global__ void __launch_bounds__(kThreads)      // (kThreads, 8) = 32 registers spills 40 bytes: 23.5 -> 28.2 us per image
warp_nhwc3_kernel(const float* __restrict__ src, const float* __restrict__ flow, float* __restrict__ dst,
                  const float* __restrict__ ref, float* __restrict__ norm_out,
                  int64_t n_pix, int H, int W, int bilinear, int vec_store, const PixDecode pd,
                  int skip, int ref_shared, int64_t win_src) {
  // skip >= 0 (window mode): batch item b samples image b of `src` when b < skip, else image b+1 -- the
  // neighbours of a frame window with the centre frame left out, no gathered copy of the frames needed;
  // ref_shared: every batch item is compared with the SAME reference image (the centre frame).
  // blockIdx.y: the frame window (src and ref advance by win_src floats per window, flow / dst / norm_out by the
  // window's n_pix pixels); a single-window launch has gridDim.y == 1.
  if (blockIdx.y) {
    const int64_t wb = blockIdx.y;
    src += wb * win_src;
    flow += wb * n_pix * 2;
    dst += wb * n_pix * 3;
    if (ref) ref += wb * win_src;
    if (norm_out) norm_out += wb * n_pix;
  }
  // two staging buffers, used alternately: one barrier per iteration (the barrier of iteration k+1 separates the
  // reads of buffer k & 1 from its next writes in iteration k+2)
  __shared__ __align__(16) float stage2[2][kThreads * 3];
  int buf = 0;
  const int64_t HW = (int64_t)H * W;
  // the flow of the NEXT iteration's pixel is loaded one iteration ahead: the taps depend on it, and with the load
  // inside the iteration every pixel paid two DRAM latencies back to back (flow, then taps) with 8 bytes in flight
  // per thread during the first
  const int64_t step = (int64_t)gridDim.x * kThreads;
  float2 f_next = make_float2(0.f, 0.f);
  {
    const int64_t i0 = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i0 < n_pix) f_next = ldg_stream_f2(reinterpret_cast<const float2*>(flow) + i0);
  }
  for (int64_t base = (int64_t)blockIdx.x * kThreads; base < n_pix; base += step, buf ^= 1) {
    float* stage = stage2[buf];
    int64_t i = base + threadIdx.x;
    float v0 = 0.f, v1 = 0.f, v2 = 0.f;
    const float2 f = f_next;
    if (i + step < n_pix) f_next = ldg_stream_f2(reinterpret_cast<const float2*>(flow) + i + step);
    if (i < n_pix) {
      int x, y, bi;
      decode_pix((uint32_t)i, pd, bi, y, x);
      const int64_t b = bi;
      const float* s = src + (b + ((skip >= 0 && bi >= skip) ? 1 : 0)) * HW * 3;
      if (bilinear) {
        Taps t = bilinear_taps<FAST>(x, y, f.x, f.y, W, H);
        const float* pTL = s + ((int64_t)t.yT * W + t.xL) * 3;
        const float* pTR = s + ((int64_t)t.yT * W + t.xR) * 3;
        const float* pBL = s + ((int64_t)t.yB * W + t.xL) * 3;
        const float* pBR = s + ((int64_t)t.yB * W + t.xR) * 3;
        v0 = blend_mode<FAST>(t, __ldg(pTL + 0), __ldg(pTR + 0), __ldg(pBL + 0), __ldg(pBR + 0));
        v1 = blend_mode<FAST>(t, __ldg(pTL + 1), __ldg(pTR + 1), __ldg(pBL + 1), __ldg(pBR + 1));
        v2 = blend_mode<FAST>(t, __ldg(pTL + 2), __ldg(pTR + 2), __ldg(pBL + 2), __ldg(pBR + 2));
      } else {
        int xN, yN;
        nearest_tap(x, y, f.x, f.y, W, H, xN, yN);
        const float* p = s + ((int64_t)yN * W + xN) * 3;
        v0 = __ldg(p);
        v1 = __ldg(p + 1);
        v2 = __ldg(p + 2);
      }
      if (norm_out != nullptr) {
        // channelnorm_kernel.cu:53-59: fp32 `result += val*val` (an FMA under nvcc's default
        // contraction) in channel order, then sqrt.
        const float* r = ref + (ref_shared ? (i - b * HW) : i) * 3;
        float d0 = __fsub_rn(__ldg(r), v0), d1 = __fsub_rn(__ldg(r + 1), v1), d2 = __fsub_rn(__ldg(r + 2), v2);
        float acc = fmaf(d0, d0, 0.0f);
        acc = fmaf(d1, d1, acc);
        acc = fmaf(d2, d2, acc);
        norm_out[i] = sqrtf(acc);
      }
    }
    stage[threadIdx.x * 3 + 0] = v0;
    stage[threadIdx.x * 3 + 1] = v1;
    stage[threadIdx.x * 3 + 2] = v2;
    __syncthreads();
    int64_t n_here = min((int64_t)kThreads, n_pix - base) * 3;  // floats owned by this block
    float* out = dst + base * 3;
    if (vec_store) {
      int n4 = (int)(n_here / 4);
      for (int k = threadIdx.x; k < n4; k += kThreads)
        stg_stream_f4(reinterpret_cast<float4*>(out) + k, reinterpret_cast<const float4*>(stage)[k]);
      for (int k = n4 * 4 + threadIdx.x; k < n_here; k += kThreads) out[k] = stage[k];
    } else {
      for (int k = threadIdx.x; k < n_here; k += kThreads) out[k] = stage[k];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Channels-last, C % 4 == 0 (features).  One thread per (pixel, 4-channel group): four 16-byte
// gathers and one 16-byte coalesced store; the C/4 lanes of a pixel share taps through the
// broadcast of the flow load.
// ---------------------------------------------------------------------------------------------
template <bool FAST>
__global__ void __launch_bounds__(kThreads)
warp_nhwc_vec4_kernel(const float* __restrict__ src, const float* __restrict__ flow, float* __restrict__ dst,
                      int64_t n_pix, int H, int W, int C, int bilinear, const PixDecode pd, const FastDiv gd) {
  const int G = C >> 2;
  const int64_t HW = (int64_t)H * W;
  const int64_t n = n_pix * G;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = fdiv((uint32_t)j, gd);
    int g = (int)(j - i * G);
    int x, y, bi;
    decode_pix((uint32_t)i, pd, bi, y, x);
    const int64_t b = bi;
    float2 f = __ldg(reinterpret_cast<const float2*>(flow) + i);
    const float4* s = reinterpret_cast<const float4*>(src + b * HW * C) + g;
    float4 o;
    if (bilinear) {
      Taps t = bilinear_taps<FAST>(x, y, f.x, f.y, W, H);
      float4 tl = __ldg(s + ((int64_t)t.yT * W + t.xL) * G);
      float4 tr = __ldg(s + ((int64_t)t.yT * W + t.xR) * G);
      float4 bl = __ldg(s + ((int64_t)t.yB * W + t.xL) * G);
      float4 br = __ldg(s + ((int64_t)t.yB * W + t.xR) * G);
      o.x = blend_mode<FAST>(t, tl.x, tr.x, bl.x, br.x);
      o.y = blend_mode<FAST>(t, tl.y, tr.y, bl.y, br.y);
      o.z = blend_mode<FAST>(t, tl.z, tr.z, bl.z, br.z);
      o.w = blend_mode<FAST>(t, tl.w, tr.w, bl.w, br.w);
    } else {
      int xN, yN;
      nearest_tap(x, y, f.x, f.y, W, H, xN, yN);
      o = __ldg(s + ((int64_t)yN * W + xN) * G);
    }
    stg_stream_f4(reinterpret_cast<float4*>(dst) + j, o);
  }
}

// Channels-last, any C: one thread per pixel, channel loop (also serves the fused norm for C != 3,
// keeping the reference's channel-order fp32 accumulation).
__global__ void __launch_bounds__(kThreads)
warp_nhwc_generic_kernel(const float* __restrict__ src, const float* __restrict__ flow, float* __restrict__ dst,
                         const float* __restrict__ ref, float* __restrict__ norm_out,
                         int64_t n_pix, int H, int W, int C, int bilinear, const PixDecode pd) {
  const int64_t HW = (int64_t)H * W;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pix; i += (int64_t)gridDim.x * blockDim.x) {
    int x, y, bi;
    decode_pix((uint32_t)i, pd, bi, y, x);
    const int64_t b = bi;
    float2 f = __ldg(reinterpret_cast<const float2*>(flow) + i);
    const float* s = src + b * HW * C;
    float* o = dst + i * C;
    float acc = 0.0f;
    if (bilinear) {
      Taps t = bilinear_taps(x, y, f.x, f.y, W, H);
      const float* pTL = s + ((int64_t)t.yT * W + t.xL) * C;
      const float* pTR = s + ((int64_t)t.yT * W + t.xR) * C;
      const float* pBL = s + ((int64_t)t.yB * W + t.xL) * C;
      const float* pBR = s + ((int64_t)t.yB * W + t.xR) * C;
      for (int c = 0; c < C; ++c) {
        float v = bilinear == kModeFast ? blend_fast(t, __ldg(pTL + c), __ldg(pTR + c), __ldg(pBL + c), __ldg(pBR + c))
                                        : blend(t, __ldg(pTL + c), __ldg(pTR + c), __ldg(pBL + c), __ldg(pBR + c));
        o[c] = v;
        if (norm_out != nullptr) {
          float d = __fsub_rn(__ldg(ref + i * C + c), v);
          acc = fmaf(d, d, acc);
        }
      }
    } else {
      int xN, yN;
      nearest_tap(x, y, f.x, f.y, W, H, xN, yN);
      const float* p = s + ((int64_t)yN * W + xN) * C;
      for (int c = 0; c < C; ++c) {
        float v = __ldg(p + c);
        o[c] = v;
        if (norm_out != nullptr) {
          float d = __fsub_rn(__ldg(ref + i * C + c), v);
          acc = fmaf(d, d, acc);
        }
      }
    }
    if (norm_out != nullptr) norm_out[i] = sqrtf(acc);
  }
}

// ---------------------------------------------------------------------------------------------
// u8 label warp (nearest).  Eight consecutive pixels per thread: four 16-byte flow loads in flight, then
// eight byte gathers in flight, one 64-bit store (with four pixels per thread -- two loads, four gathers --
// the kernel sat at 54 % of HBM waiting on its own dependent loads).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
warp_labels_kernel(const uint8_t* __restrict__ labels, const float* __restrict__ flow, uint8_t* __restrict__ dst,
                   int64_t n_pix, int H, int W, int vec, const PixDecode pd, int64_t flow_stride) {
  const int64_t HW = (int64_t)H * W;
  if (blockIdx.y) {     // window blockIdx.y: labels / dst advance by its n_pix pixels, flow by flow_stride floats
    const int64_t wb = blockIdx.y;
    labels += wb * n_pix;
    dst += wb * n_pix;
    flow += wb * flow_stride;
  }
  const int64_t n8 = vec ? n_pix / 8 : 0;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n8; q += (int64_t)gridDim.x * blockDim.x) {
    float4 f[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) f[j] = ldg_stream_f4(reinterpret_cast<const float4*>(flow) + q * 4 + j);
    const float fxs[8] = {f[0].x, f[0].z, f[1].x, f[1].z, f[2].x, f[2].z, f[3].x, f[3].z};
    const float fys[8] = {f[0].y, f[0].w, f[1].y, f[1].w, f[2].y, f[2].w, f[3].y, f[3].w};
    const uint8_t* src[8];
    int x0, y0, b0;
    decode_pix((uint32_t)(q * 8), pd, b0, y0, x0);        // one index decode per 8 pixels unless the run wraps a row
    const bool same_row = x0 + 7 < W;
    const uint8_t* img0 = labels + (int64_t)b0 * HW;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      int x = x0 + k, y = y0;
      const uint8_t* img = img0;
      if (!same_row) {
        int bi;
        decode_pix((uint32_t)(q * 8 + k), pd, bi, y, x);
        img = labels + (int64_t)bi * HW;
      }
      int xN, yN;
      nearest_tap(x, y, fxs[k], fys[k], W, H, xN, yN);
      src[k] = img + (yN * W + xN);
    }
    uint32_t v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = __ldg(src[k]);
    uint2 packed;
    packed.x = v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24);
    packed.y = v[4] | (v[5] << 8) | (v[6] << 16) | (v[7] << 24);
    reinterpret_cast<uint2*>(dst)[q] = packed;
  }
  // scalar tail (and the whole range when the buffers are not 16/4-byte aligned)
  for (int64_t i = n8 * 8 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pix;
       i += (int64_t)gridDim.x * blockDim.x) {
    int x, y, bi;
    decode_pix((uint32_t)i, pd, bi, y, x);
    const int64_t b = bi;
    float2 f = __ldg(reinterpret_cast<const float2*>(flow) + i);
    int xN, yN;
    nearest_tap(x, y, f.x, f.y, W, H, xN, yN);
    dst[i] = __ldg(labels + b * HW + (int64_t)yN * W + xN);
  }
}

// channelnorm_kernel.cu:19-60 for the other two dtypes of its AT_DISPATCH_FLOATING_TYPES_AND_HALF (:111): `val * val` is
// evaluated in scalar_t (c10::Half: float product rounded to half; double: double product), cast to float and summed
// in fp32; sqrt in fp32; the result cast back to scalar_t.
__device__ __forceinline__ float sq_as(const __half v) { return __half2float(__float2half_rn(__half2float(v) * __half2float(v))); }
__device__ __forceinline__ float sq_as(const double v) { return __double2float_rn(__dmul_rn(v, v)); }
__device__ __forceinline__ void store_as(__half* p, float v) { *p = __float2half_rn(v); }
__device__ __forceinline__ void store_as(double* p, float v) { *p = (double)v; }
__device__ __forceinline__ float load_f(const __half* p) { return __half2float(*p); }
__device__ __forceinline__ float load_f(const double* p) { return __double2float_rn(*p); }
template <typename T>
__global__ void __launch_bounds__(kThreads)
channelnorm_nchw_typed_kernel(const T* __restrict__ in, T* __restrict__ out, int B, int C, int H, int W) {
  const int64_t HW = (int64_t)H * W;
  const int64_t n = (int64_t)B * HW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / HW, p = i - b * HW;
    const T* s = in + b * C * HW + p;
    float acc = 0.0f;
    for (int c = 0; c < C; ++c) acc = __fadd_rn(acc, sq_as(s[(int64_t)c * HW]));
    store_as(out + i, sqrtf(acc));
  }
}
// channelnorm_kernel.cu:64-96: val = float(g) * float(x) / (float(out) + 1e-9) [the literal makes it a double division],
// rounded to float, cast to scalar_t
template <typename T>
__global__ void __launch_bounds__(kThreads)
channelnorm_backward_typed_kernel(const T* __restrict__ in, const T* __restrict__ out, const T* __restrict__ gout,
                                  T* __restrict__ gin, int C, int64_t HW, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / (C * HW);
    const int64_t p = i % HW;
    const int64_t oi = b * HW + p;
    const float num = __fmul_rn(load_f(gout + oi), load_f(in + i));
    store_as(gin + i, __double2float_rn(__ddiv_rn((double)num, __dadd_rn((double)load_f(out + oi), 1e-9))));
  }
}

// channelnorm_kernel.cu:19-60, NCHW: one thread per (b, y, x), coalesced plane reads.
__global__ void __launch_bounds__(kThreads)
channelnorm_nchw_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int C, int H, int W) {
  const int64_t HW = (int64_t)H * W;
  const int64_t n = (int64_t)B * HW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t b = i / HW;
    int64_t p = i - b * HW;
    const float* s = in + b * C * HW + p;
    float acc = 0.0f;
    for (int c = 0; c < C; ++c) {
      float v = __ldg(s + (int64_t)c * HW);
      acc = fmaf(v, v, acc);
    }
    out[i] = sqrtf(acc);
  }
}

// ---------------------------------------------------------------------------------------------
// Flow composition: out(p) = g(p) + f(p + g(p)), f sampled bilinearly with the warp's taps and border
// rule (fast fp32 blend).  g maps the pixels of image A to image B, f the pixels of B to C: out maps A to C.
// The pipeline chains the projected flows of the past frames / the forward flows of the future frames into
// centre -> neighbour flows with it, one image per call.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
compose_flow_kernel(const float2* __restrict__ g, const float2* __restrict__ f, float2* __restrict__ out,
                    int64_t n_pix, int H, int W, const PixDecode pd, int64_t win_stride) {
  const int64_t HW = (int64_t)H * W;
  if (blockIdx.y) {     // window blockIdx.y: g, f and out advance by win_stride flow vectors
    const int64_t o = blockIdx.y * win_stride;
    if (g) g += o;
    f += o;
    out += o;
  }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pix; i += (int64_t)gridDim.x * blockDim.x) {
    int x, y, bi;
    decode_pix((uint32_t)i, pd, bi, y, x);
    const float2 gv = g ? ldg_stream_f2(g + i) : make_float2(0.f, 0.f);   // g == NULL: the identity, out = f (a copy)
    const float2* s = f + (int64_t)bi * HW;
    const Taps t = bilinear_taps<true>(x, y, gv.x, gv.y, W, H);
    const float2 tl = __ldg(s + (int64_t)t.yT * W + t.xL), tr = __ldg(s + (int64_t)t.yT * W + t.xR);
    const float2 bl = __ldg(s + (int64_t)t.yB * W + t.xL), br = __ldg(s + (int64_t)t.yB * W + t.xR);
    out[i] = make_float2(__fadd_rn(gv.x, blend_fast(t, tl.x, tr.x, bl.x, br.x)),
                         __fadd_rn(gv.y, blend_fast(t, tl.y, tr.y, bl.y, br.y)));
  }
}

inline int grid_for(int64_t work_items, int per_block) {
  int64_t blocks = ceil_div64(work_items, per_block);
  // enough CTAs for every SM to hold its full complement of 256-thread blocks (8/SM), a whole
  // number of waves; grid-stride loops absorb the rest.
  int64_t cap = (int64_t)kNumSMs * 8 * 4;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

inline bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

}  // namespace
}  // namespace vsr

using namespace vsr;

extern "C" int vsr_resample2d_forward(const float* input1, const float* flow, float* output, int B, int C, int H,
                                      int W, int kernel_size, int bilinear, vsr_stream_t stream) {
  if (!input1 || !flow || !output || B <= 0 || C <= 0 || H <= 0 || W <= 0) return VSR_ERR_INVALID_ARG;
  if (kernel_size < 1 || kernel_size > 16) return VSR_ERR_UNSUPPORTED;  // resample2d.py:44 only ever uses 1
  int64_t n = (int64_t)B * H * W;
  if (n >= ((int64_t)1 << 32)) return VSR_ERR_UNSUPPORTED;   // 32-bit index decode
  resample2d_nchw_kernel<<<grid_for(n, kThreads), kThreads, 0, as_stream(stream)>>>(input1, flow, output, B, C, H, W,
                                                                                   bilinear ? 1 : 0, make_pixdecode(H, W),
                                                                                   kernel_size);
  return after_launch();
}

extern "C" int vsr_warp_nhwc_f32(const float* src, const float* flow, float* dst, const float* ref, float* norm_out,
                                 int B, int H, int W, int C, int bilinear, vsr_stream_t stream) {
  if (!src || !flow || !dst || B <= 0 || C <= 0 || H <= 0 || W <= 0) return VSR_ERR_INVALID_ARG;
  if ((norm_out != nullptr) != (ref != nullptr)) return VSR_ERR_INVALID_ARG;
  if (!aligned(flow, 8)) return VSR_ERR_INVALID_ARG;
  int64_t n_pix = (int64_t)B * H * W;
  cudaStream_t st = as_stream(stream);
  if (bilinear < 0 || bilinear > kModeFast) return VSR_ERR_INVALID_ARG;
  if ((int64_t)B * H * W * ((C % 4) == 0 ? C / 4 : 1) >= ((int64_t)1 << 32)) return VSR_ERR_UNSUPPORTED;   // 32-bit index decode
  const PixDecode pd = make_pixdecode(H, W);
  if (C == 3) {
    // (a 4-pixels-per-thread variant without the shared-memory staging measured SLOWER on B200, 195 vs
    //  172 us for 8 x 1080p: neighbouring lanes' gathers end up 48 B apart and touch 4x more lines per load)
    int vec = aligned(dst, 16) ? 1 : 0;
    if (bilinear == kModeFast)
      warp_nhwc3_kernel<true><<<grid_for(n_pix, kThreads), kThreads, 0, st>>>(src, flow, dst, ref, norm_out, n_pix, H, W,
                                                                              1, vec, pd, -1, 0, 0);
    else
      warp_nhwc3_kernel<false><<<grid_for(n_pix, kThreads), kThreads, 0, st>>>(src, flow, dst, ref, norm_out, n_pix, H,
                                                                               W, bilinear, vec, pd, -1, 0, 0);
  } else if ((C % 4) == 0 && norm_out == nullptr && aligned(src, 16) && aligned(dst, 16)) {
    if (bilinear == kModeFast)
      warp_nhwc_vec4_kernel<true><<<grid_for(n_pix * (C / 4), kThreads), kThreads, 0, st>>>(src, flow, dst, n_pix, H, W,
                                                                                            C, 1, pd, make_fastdiv((uint32_t)(C / 4)));
    else
      warp_nhwc_vec4_kernel<false><<<grid_for(n_pix * (C / 4), kThreads), kThreads, 0, st>>>(src, flow, dst, n_pix, H,
                                                                                             W, C, bilinear, pd, make_fastdiv((uint32_t)(C / 4)));
  } else {
    warp_nhwc_generic_kernel<<<grid_for(n_pix, kThreads), kThreads, 0, st>>>(src, flow, dst, ref, norm_out, n_pix, H,
                                                                             W, C, bilinear, pd);
  }
  return after_launch();
}

extern "C" int vsr_warp_windows_nhwc3(const float* frames, const float* flows, float* warped, float* resid, int windows,
                                      int T, int centre, int H, int W, int bilinear, vsr_stream_t stream) {
  if (!frames || !flows || !warped || windows < 1 || windows > 65535 || T < 2 || centre < 0 || centre >= T || H <= 0 ||
      W <= 0)
    return VSR_ERR_INVALID_ARG;
  if (bilinear < 0 || bilinear > kModeFast || !aligned(flows, 8)) return VSR_ERR_INVALID_ARG;
  const int64_t n_pix = (int64_t)(T - 1) * H * W;     // per window
  if (n_pix >= ((int64_t)1 << 32)) return VSR_ERR_UNSUPPORTED;
  const PixDecode pd = make_pixdecode(H, W);
  const float* ref = resid ? frames + (int64_t)centre * H * W * 3 : nullptr;
  // 16-byte stores need every window's output to start 16-byte aligned
  const int vec = aligned(warped, 16) && (windows == 1 || (n_pix * 3) % 4 == 0) ? 1 : 0;
  const int64_t win_src = (int64_t)T * H * W * 3;
  const dim3 grid(grid_for(n_pix, kThreads), windows);
  cudaStream_t st = as_stream(stream);
  if (bilinear == kModeFast)
    warp_nhwc3_kernel<true><<<grid, kThreads, 0, st>>>(frames, flows, warped, ref, resid, n_pix, H, W, 1, vec, pd, centre,
                                                       1, win_src);
  else
    warp_nhwc3_kernel<false><<<grid, kThreads, 0, st>>>(frames, flows, warped, ref, resid, n_pix, H, W, bilinear, vec, pd,
                                                        centre, 1, win_src);
  return after_launch();
}

extern "C" int vsr_compose_flow_windows(const float* g, const float* f, float* out, int windows, int64_t stride, int H,
                                        int W, vsr_stream_t stream) {
  if (!f || !out || windows < 1 || windows > 65535 || stride < 0 || (stride & 1) || H <= 0 || W <= 0)
    return VSR_ERR_INVALID_ARG;
  if (!aligned(g, 8) || !aligned(f, 8) || !aligned(out, 8)) return VSR_ERR_INVALID_ARG;
  const int64_t n_pix = (int64_t)H * W;
  if (n_pix >= ((int64_t)1 << 32)) return VSR_ERR_UNSUPPORTED;
  compose_flow_kernel<<<dim3(grid_for(n_pix, kThreads), windows), kThreads, 0, as_stream(stream)>>>(
      reinterpret_cast<const float2*>(g), reinterpret_cast<const float2*>(f), reinterpret_cast<float2*>(out), n_pix, H, W,
      make_pixdecode(H, W), stride / 2);
  return after_launch();
}

extern "C" int vsr_warp_labels_u8(const uint8_t* labels, const float* flow, uint8_t* dst, int B, int H, int W,
                                  vsr_stream_t stream) {
  if (!labels || !flow || !dst || B <= 0 || H <= 0 || W <= 0) return VSR_ERR_INVALID_ARG;
  if (!aligned(flow, 8)) return VSR_ERR_INVALID_ARG;
  int64_t n_pix = (int64_t)B * H * W;
  if (n_pix >= ((int64_t)1 << 32)) return VSR_ERR_UNSUPPORTED;   // 32-bit index decode
  int vec = (aligned(flow, 16) && aligned(dst, 8)) ? 1 : 0;
  warp_labels_kernel<<<grid_for(ceil_div64(n_pix, 8), kThreads), kThreads, 0, as_stream(stream)>>>(labels, flow, dst,
                                                                                                  n_pix, H, W, vec, make_pixdecode(H, W), 0);
  return after_launch();
}

extern "C" int vsr_warp_labels_u8_windows(const uint8_t* labels, const float* flow, uint8_t* dst, int windows,
                                          int64_t flow_stride, int H, int W, vsr_stream_t stream) {
  if (!labels || !flow || !dst || windows < 1 || windows > 65535 || flow_stride < 0 || H <= 0 || W <= 0)
    return VSR_ERR_INVALID_ARG;
  if (!aligned(flow, 8) || (flow_stride & 1)) return VSR_ERR_INVALID_ARG;
  const int64_t n_pix = (int64_t)H * W;     // per window
  if (n_pix >= ((int64_t)1 << 32)) return VSR_ERR_UNSUPPORTED;
  // the vector path needs every window's flow 16-byte and output 8-byte aligned
  const int vec = (aligned(flow, 16) && aligned(dst, 8) && (windows == 1 || (flow_stride % 4 == 0 && n_pix % 8 == 0)))
                      ? 1 : 0;
  warp_labels_kernel<<<dim3(grid_for(ceil_div64(n_pix, 8), kThreads), windows), kThreads, 0, as_stream(stream)>>>(
      labels, flow, dst, n_pix, H, W, vec, make_pixdecode(H, W), flow_stride);
  return after_launch();
}

extern "C" int vsr_channelnorm_forward(const float* input, float* output, int B, int C, int H, int W, int norm_deg,
                                       vsr_stream_t stream) {
  (void)norm_deg;  // accepted and ignored, as channelnorm_kernel.cu:53-59 does
  if (!input || !output || B <= 0 || C <= 0 || H <= 0 || W <= 0) return VSR_ERR_INVALID_ARG;
  int64_t n = (int64_t)B * H * W;
  channelnorm_nchw_kernel<<<grid_for(n, kThreads), kThreads, 0, as_stream(stream)>>>(input, output, B, C, H, W);
  return after_launch();
}

// ---------------------------------------------------------------------------------------------
// Backward passes (SURVEY.md 8f rank 2): complete the autograd Function surfaces.
//   ref: resample2d_kernel.cu:75-125 (gradient w.r.t. input1: 4-tap scatter with atomicAdd),
//        :127-198 (gradient w.r.t. the flow), channelnorm_kernel.cu:64-96.
// The reference's quirks are kept: the scatter's fractional parts use int() truncation, not floor
// (:105-106), its taps use floor (:111-114), `bilinear` is ignored, kernel_size must be 1.
// ---------------------------------------------------------------------------------------------
namespace vsr {
namespace {

__device__ __forceinline__ void red_add_f32(float* addr, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(addr), "f"(v) : "memory");
}

// One thread per (b, y, x): taps and weights once, then the channel loop (the reference spends one
// thread per (b, c, y, x) and recomputes them C times).
__global__ void __launch_bounds__(kThreads)
resample2d_backward_input1_kernel(const float* __restrict__ flow, const float* __restrict__ gout, float* __restrict__ gin1,
                                  int B, int C, int H, int W, const PixDecode pd) {
  const int64_t HW = (int64_t)H * W;
  const int64_t n = (int64_t)B * HW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int x, y, b;
    decode_pix((uint32_t)i, pd, b, y, x);
    const float* fl = flow + (int64_t)b * 2 * HW + (int64_t)y * W + x;
    const float dx = __ldg(fl), dy = __ldg(fl + HW);
    const float xf = __fadd_rn((float)x, dx), yf = __fadd_rn((float)y, dy);
    const float alpha = __fsub_rn(xf, (float)__float2int_rz(xf));     // :105 int(), not floor
    const float beta = __fsub_rn(yf, (float)__float2int_rz(yf));      // :106
    const int xL = max(min((int)floorf(xf), W - 1), 0);
    const int xR = max(min((int)__fadd_rn(floorf(xf), 1.0f), W - 1), 0);
    const int yT = max(min((int)floorf(yf), H - 1), 0);
    const int yB = max(min((int)__fadd_rn(floorf(yf), 1.0f), H - 1), 0);
    const float ia = __fsub_rn(1.0f, alpha), ib = __fsub_rn(1.0f, beta);
    const float wTL = __fmul_rn(ia, ib), wTR = __fmul_rn(alpha, ib), wBL = __fmul_rn(ia, beta), wBR = __fmul_rn(alpha, beta);
    const int64_t oTL = (int64_t)yT * W + xL, oTR = (int64_t)yT * W + xR, oBL = (int64_t)yB * W + xL, oBR = (int64_t)yB * W + xR;
    for (int c = 0; c < C; ++c) {
      const float g = __ldg(gout + ((int64_t)b * C + c) * HW + (int64_t)y * W + x);
      float* plane = gin1 + ((int64_t)b * C + c) * HW;
      red_add_f32(plane + oTL, __fmul_rn(wTL, g));
      red_add_f32(plane + oTR, __fmul_rn(wTR, g));
      red_add_f32(plane + oBL, __fmul_rn(wBL, g));
      red_add_f32(plane + oBR, __fmul_rn(wBR, g));
    }
  }
}

// One thread per (b, y, x) computes both flow-gradient channels (the reference: one thread per
// channel, each re-reading the C taps).  The accumulation order and the FMA contraction of
// `output += gamma * g * in` are the reference binary's, so the result is bit-identical.
__global__ void __launch_bounds__(kThreads)
resample2d_backward_input2_kernel(const float* __restrict__ in1, const float* __restrict__ flow,
                                  const float* __restrict__ gout, float* __restrict__ gin2, int B, int C, int H, int W,
                                  const PixDecode pd) {
  const int64_t HW = (int64_t)H * W;
  const int64_t n = (int64_t)B * HW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int x, y, b;
    decode_pix((uint32_t)i, pd, b, y, x);
    const float* fl = flow + (int64_t)b * 2 * HW + (int64_t)y * W + x;
    const float dx = __ldg(fl), dy = __ldg(fl + HW);
    const float xf = __fadd_rn((float)x, dx), yf = __fadd_rn((float)y, dy);
    const float fx0 = floorf(xf), fy0 = floorf(yf);
    const int xL = max(min((int)fx0, W - 1), 0);
    const int xR = max(min((int)__fadd_rn(fx0, 1.0f), W - 1), 0);
    const int yT = max(min((int)fy0, H - 1), 0);
    const int yB = max(min((int)__fadd_rn(fy0, 1.0f), H - 1), 0);
    const float gx = __fsub_rn(1.0f, __fsub_rn(yf, fy0));   // channel 0 (dx): gamma = 1 - (yf - floor(yf)), :179
    const float gy = __fsub_rn(1.0f, __fsub_rn(xf, fx0));   // channel 1 (dy): gamma = 1 - (xf - floor(xf)), :166
    const float igx = __fsub_rn(1.0f, gx), igy = __fsub_rn(1.0f, gy);
    const int64_t oTL = (int64_t)yT * W + xL, oTR = (int64_t)yT * W + xR, oBL = (int64_t)yB * W + xL, oBR = (int64_t)yB * W + xR;
    float out0 = 0.0f, out1 = 0.0f;
    for (int ch = 0; ch < C; ++ch) {
      const float g = __ldg(gout + ((int64_t)b * C + ch) * HW + (int64_t)y * W + x);
      const float* p = in1 + ((int64_t)b * C + ch) * HW;
      const float tl = __ldg(p + oTL), tr = __ldg(p + oTR), bl = __ldg(p + oBL), br = __ldg(p + oBR);
      // c % 2 == 0 (:178-189): +g*TR -g*TL +(1-g)*BR -(1-g)*BL
      const float a0 = __fmul_rn(gx, g), b0 = __fmul_rn(igx, g);
      out0 = fmaf(a0, tr, out0);
      out0 = fmaf(-a0, tl, out0);
      out0 = fmaf(b0, br, out0);
      out0 = fmaf(-b0, bl, out0);
      // c % 2 == 1 (:165-176): +g*BL -g*TL +(1-g)*BR -(1-g)*TR
      const float a1 = __fmul_rn(gy, g), b1 = __fmul_rn(igy, g);
      out1 = fmaf(a1, bl, out1);
      out1 = fmaf(-a1, tl, out1);
      out1 = fmaf(b1, br, out1);
      out1 = fmaf(-b1, tr, out1);
    }
    float* o = gin2 + (int64_t)b * 2 * HW + (int64_t)y * W + x;
    o[0] = out0;
    o[HW] = out1;
  }
}

// channelnorm_kernel.cu:64-96: val = float(g * x) / (double(out) + 1e-9), rounded to fp32
__global__ void __launch_bounds__(kThreads)
channelnorm_backward_kernel(const float* __restrict__ in, const float* __restrict__ out, const float* __restrict__ gout,
                            float* __restrict__ gin, int C, int64_t HW, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / (C * HW);
    const int64_t p = i % HW;
    const int64_t oi = b * HW + p;
    const float num = __fmul_rn(__ldg(gout + oi), __ldg(in + i));
    gin[i] = __double2float_rn(__ddiv_rn((double)num, __dadd_rn((double)__ldg(out + oi), 1e-9)));
  }
}

}  // namespace

int launch_resample2d_backward_input2(const float* input1, const float* flow, const float* grad_output,
                                      float* grad_input2, int B, int C, int H, int W, cudaStream_t st) {
  const int64_t n = (int64_t)B * H * W;
  resample2d_backward_input2_kernel<<<grid_for(n, kThreads), kThreads, 0, st>>>(input1, flow, grad_output, grad_input2, B, C,
                                                                               H, W, make_pixdecode(H, W));
  return after_launch();
}

}  // namespace vsr

extern "C" int vsr_resample2d_backward(const float* input1, const float* flow, const float* grad_output,
                                       float* grad_input1, float* grad_input2, int B, int C, int H, int W,
                                       int kernel_size, int bilinear, vsr_stream_t stream) {
  (void)bilinear;  // the reference's backward ignores it as well (resample2d_kernel.cu:75-198)
  if (!input1 || !flow || !grad_output || !grad_input1 || !grad_input2 || B <= 0 || C <= 0 || H <= 0 || W <= 0)
    return VSR_ERR_INVALID_ARG;
  if (kernel_size != 1) return VSR_ERR_UNSUPPORTED;
  if ((int64_t)B * H * W >= ((int64_t)1 << 32)) return VSR_ERR_UNSUPPORTED;
  const int64_t n = (int64_t)B * H * W;
  const PixDecode pd = make_pixdecode(H, W);
  cudaStream_t st = as_stream(stream);
  resample2d_backward_input1_kernel<<<grid_for(n, kThreads), kThreads, 0, st>>>(flow, grad_output, grad_input1, B, C, H, W, pd);
  int rc = after_launch();
  if (rc) return rc;
  return launch_resample2d_backward_input2(input1, flow, grad_output, grad_input2, B, C, H, W, st);
}

extern "C" int vsr_channelnorm_forward_typed(const void* input, void* output, int B, int C, int H, int W, int norm_deg,
                                             int dtype, vsr_stream_t stream) {
  (void)norm_deg;
  if (dtype == VSR_DTYPE_F32)
    return vsr_channelnorm_forward(static_cast<const float*>(input), static_cast<float*>(output), B, C, H, W, norm_deg, stream);
  if (!input || !output || B <= 0 || C <= 0 || H <= 0 || W <= 0) return VSR_ERR_INVALID_ARG;
  const int64_t n = (int64_t)B * H * W;
  cudaStream_t st = as_stream(stream);
  if (dtype == VSR_DTYPE_F16)
    channelnorm_nchw_typed_kernel<__half><<<grid_for(n, kThreads), kThreads, 0, st>>>(static_cast<const __half*>(input),
                                                                                  static_cast<__half*>(output), B, C, H, W);
  else if (dtype == VSR_DTYPE_F64)
    channelnorm_nchw_typed_kernel<double><<<grid_for(n, kThreads), kThreads, 0, st>>>(static_cast<const double*>(input),
                                                                                  static_cast<double*>(output), B, C, H, W);
  else
    return VSR_ERR_UNSUPPORTED;
  return after_launch();
}

extern "C" int vsr_channelnorm_backward_typed(const void* input, const void* output, const void* grad_output,
                                              void* grad_input, int B, int C, int H, int W, int norm_deg, int dtype,
                                              vsr_stream_t stream) {
  if (dtype == VSR_DTYPE_F32)
    return vsr_channelnorm_backward(static_cast<const float*>(input), static_cast<const float*>(output),
                                    static_cast<const float*>(grad_output), static_cast<float*>(grad_input), B, C, H, W,
                                    norm_deg, stream);
  if (!input || !output || !grad_output || !grad_input || B <= 0 || C <= 0 || H <= 0 || W <= 0) return VSR_ERR_INVALID_ARG;
  const int64_t HW = (int64_t)H * W, n = (int64_t)B * C * HW;
  cudaStream_t st = as_stream(stream);
  if (dtype == VSR_DTYPE_F16)
    channelnorm_backward_typed_kernel<__half><<<grid_for(n, kThreads), kThreads, 0, st>>>(
        static_cast<const __half*>(input), static_cast<const __half*>(output), static_cast<const __half*>(grad_output),
        static_cast<__half*>(grad_input), C, HW, n);
  else if (dtype == VSR_DTYPE_F64)
    channelnorm_backward_typed_kernel<double><<<grid_for(n, kThreads), kThreads, 0, st>>>(
        static_cast<const double*>(input), static_cast<const double*>(output), static_cast<const double*>(grad_output),
        static_cast<double*>(grad_input), C, HW, n);
  else
    return VSR_ERR_UNSUPPORTED;
  return after_launch();
}

extern "C" int vsr_channelnorm_backward(const float* input, const float* output, const float* grad_output,
                                        float* grad_input, int B, int C, int H, int W, int norm_deg, vsr_stream_t stream) {
  (void)norm_deg;
  if (!input || !output || !grad_output || !grad_input || B <= 0 || C <= 0 || H <= 0 || W <= 0) return VSR_ERR_INVALID_ARG;
  const int64_t HW = (int64_t)H * W, n = (int64_t)B * C * HW;
  channelnorm_backward_kernel<<<grid_for(n, kThreads), kThreads, 0, as_stream(stream)>>>(input, output, grad_output,
                                                                                        grad_input, C, HW, n);
  return after_launch();
}
