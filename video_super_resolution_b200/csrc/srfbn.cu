// srfbn.cu -- host side of the fusion / upsampling convolution stack (a6/a7): plan, weight packing,
// TMA tensor maps and the launch sequence over the tcgen05 implicit-GEMM kernel (igemm.cuh), plus
// the two small SIMT kernels around it (input im2col, per-pixel fc fuse over the map axis).
//
//   ref: my_packages/SRProjection/SRProjectionModule.py:96-150 (SRProjectionModule),
//        :7-93 (FeedbackBlock), my_packages/SRProjection/blocks.py:7-74
//   dataflow: the INTENDED dense-concat dataflow of SURVEY.md Appendix C (the reference stages its
//   concats through torch.empty buffers it never fills, SRProjectionModule.py:55-59,70-74).
//
// Every dense layer is one launch of igemm_kernel (BF16 operands, FP32 accumulation in TMEM):
//   conv_in 3x3 3->128    : im2col'd input (K padded 27->32), pointwise GEMM, N=128
//   1x1 convs             : pointwise GEMM over up to 6 concatenated 32-channel sources (the
//                           torch.cat never materialises), N=32
//   ConvTranspose 8x8 s4  : output-stationary: block (Yb,Xb) of the "HR block layout" gets 2x2 LR
//                           taps, N = 16 sub-positions x 32 channels (two N=256 halves)
//   Conv 8x8 s4           : fused with the 1x1 "downtran" in front of it (fused_down.cuh), output-shift form
//   x2 geometry (k6 s2 p2): layered on plain NHWC HR features (build_deconv2 / build_downconv2)
//   conv_out 3x3 32->3    : 9 taps at HR, N=16 (3 used), epilogue adds the bilinear skip and the
//                           mean shifts and writes fp32 planes
// HR block layout: an HR feature map of (4h,4w) pixels is stored as (h+1, w+1) blocks of 4x4 pixels
// whose origin is shifted by (-2,-2): block (Yb,Xb), sub-position s=ry*4+rx holds HR pixel
// (4Yb+ry-2, 4Xb+rx-2); positions outside the image are a zero ring.  With this shift both 8x8-s4
// operators touch exactly 2x2 blocks (padding 2 is absorbed by the ring), and a block is one
// contiguous 1 KB row of 16 x 32 BF16.
//
// The `out` deconv and `conv_out` are evaluated for the last feedback step only: the reference
// keeps `outs[-1:]` (SRProjectionModule.py:145), the earlier steps' images are dead values.
#include "fused_down.cuh"

#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

namespace vsr {
namespace {

constexpr int kNF = 32;        // num_features
constexpr int kGroups = 6;
constexpr int kMaxMaps = 64;   // fc in-features bound (weights live in shared memory)

// ------------------------------------------------------------------------------------------------
// driver entry point (no link-time dependency on libcuda: the library must load on a CPU-only box)
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// channels-last BF16 activation tensor (b, y, x, c), c innermost; box = [ck, tw, th, 1]
int make_act_map(CUtensorMap* m, const void* base, int64_t C, int64_t W, int64_t H, int64_t B, int ck, int tw, int th) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return VSR_ERR_STATE;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)C * 2 * W, (cuuint64_t)C * 2 * W * H};
  cuuint32_t box[4] = {(cuuint32_t)ck, (cuuint32_t)tw, (cuuint32_t)th, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, ck == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? VSR_OK : VSR_ERR_CUDA_BASE + 999;
}

// packed weights [N rows][K] BF16, K innermost; box = [ck, bn]
int make_w_map(CUtensorMap* m, const void* base, int64_t K, int64_t N, int ck, int bn) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return VSR_ERR_STATE;
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)N};
  cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {(cuuint32_t)ck, (cuuint32_t)bn};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, ck == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? VSR_OK : VSR_ERR_CUDA_BASE + 999;
}

// ------------------------------------------------------------------------------------------------
// kernel variants
// ------------------------------------------------------------------------------------------------
enum Variant : int { V_PW32 = 0, V_PW128, V_DECONV, V_CONVOUT, V_FUSED_TRAN, V_FUSED_PLAIN, V_FINALIZE, V_DECONV2, V_DOWN2, V_FUSED_UPDOWN, V_COUNT };

// kernel classes for the per-launch accounting bench.py reads (vsr_srfbn_profile_*)
static_assert(VSR_SRFBN_KERNEL_CLASSES == 10, "header constant");
enum KClass : int { KC_IM2COL = 0, KC_CONV_IN, KC_PW_LR, KC_PW_HR, KC_DECONV, KC_DOWNCONV, KC_CONV_OUT, KC_FC, KC_FUSED_DOWN, KC_FINALIZE, KC_COUNT };

struct Layer {
  int variant;
  IgemmParams p;
  FusedDownParams f;     // V_FUSED_*
  float* fin_acc;        // V_FINALIZE
  const float* fin_bias;
  void* fin_out;
  int64_t fin_n8;
  int fin_w, fin_h, fin_b;
  int grid;
  size_t smem;
  int kclass;
  double flops;   // 2*MAC of the layer as specified (padding / ring rows not counted)
  double bytes;   // compulsory HBM bytes of this launch: its inputs + outputs, each once
};

template <int MODE, int CK, int BN>
int launch_variant(const Layer& L, cudaStream_t st) {
  static PerDeviceOnce once;       // the attribute is sticky per function and device
  int dev;
  if (once.needed(&dev)) {
    cudaError_t e = cudaFuncSetAttribute(igemm_kernel<MODE, CK, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         227 * 1024);
    if (e != cudaSuccess) return cuda_status(e);
    once.mark(dev);
  }
  igemm_kernel<MODE, CK, BN><<<L.grid, igemm_threads(MODE), L.smem, st>>>(L.p);
  return after_launch();
}

template <bool HAS_TRAN>
int launch_fused(const Layer& L, cudaStream_t st) {
  static PerDeviceOnce once;
  int dev;
  if (once.needed(&dev)) {
    cudaError_t e = cudaFuncSetAttribute(fused_down_kernel<HAS_TRAN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         227 * 1024);
    if (e != cudaSuccess) return cuda_status(e);
    once.mark(dev);
  }
  fused_down_kernel<HAS_TRAN><<<L.grid, kFusedThreads, L.smem, st>>>(L.f);
  return after_launch();
}

int launch_fused_updown(const Layer& L, cudaStream_t st) {
  static PerDeviceOnce once;
  int dev;
  if (once.needed(&dev)) {
    cudaError_t e = cudaFuncSetAttribute(fused_updown_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return cuda_status(e);
    once.mark(dev);
  }
  fused_updown_kernel<<<L.grid, kFusedThreads, L.smem, st>>>(L.f);
  return after_launch();
}

int launch_layer(const Layer& L, cudaStream_t st) {
  switch (L.variant) {
    case V_FUSED_UPDOWN: return launch_fused_updown(L, st);
    case V_FUSED_TRAN: return launch_fused<true>(L, st);
    case V_FUSED_PLAIN: return launch_fused<false>(L, st);
    case V_FINALIZE: {
      const int R = L.fin_h / kFinalizePeriod;
      const int64_t items = ((int64_t)L.fin_b * R * L.fin_w + (int64_t)L.fin_b * (L.fin_h - R) * (L.fin_w / 16)) * 4;
      if (items == 0) return VSR_OK;
      int64_t blocks = ceil_div64(items, 256);
      if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
      finalize_lr_kernel<<<(int)blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(L.fin_acc), L.fin_bias,
                                                      reinterpret_cast<uint4*>(L.fin_out), L.fin_b, L.fin_h, L.fin_w);
      return after_launch();
    }
    case V_PW32: return launch_variant<EPI_ROWS, 32, 32>(L, st);
    case V_PW128: return launch_variant<EPI_ROWS, 32, 128>(L, st);
    case V_DECONV: return launch_variant<EPI_DECONV, 32, 256>(L, st);
    case V_CONVOUT: return launch_variant<EPI_CONV_OUT, 32, 32>(L, st);
    case V_DECONV2: return launch_variant<EPI_DECONV2, 32, 128>(L, st);
    case V_DOWN2: return launch_variant<EPI_DOWN2, 64, 96>(L, st);
    default: return VSR_ERR_INVALID_ARG;
  }
}

size_t variant_smem(int variant, int chunks, size_t ring) {
  switch (variant) {
    case V_PW32: return igemm_smem_bytes<32, 32>(chunks, ring);
    case V_PW128: return igemm_smem_bytes<32, 128>(chunks, ring);
    case V_DECONV2: return igemm_smem_bytes<32, 128>(chunks, ring, kDeconv2StageBytes);
    case V_DECONV: return igemm_smem_bytes<32, 256>(chunks, ring, kDeconvStageBytes);
    case V_DOWN2: return igemm_smem_bytes<64, 96>(chunks, ring);
    default: return igemm_smem_bytes<32, 32>(chunks, ring, kConvOutStageBytes);
  }
}

void finish_layer(Layer& L, int ctas_per_sm) {
  IgemmParams& p = L.p;
  if (p.cps < 1) p.cps = 1;
  if (p.stage_bytes == 0) {   // default: every chunk loads its own [128 x 32] box
    constexpr int kA = a_stage_bytes<32>();
    p.stage_bytes = p.cps * kA;
    for (int i = 0; i < p.num_chunks; ++i) {
      p.chunks[i].a_off = (i % p.cps) * kA;
      p.chunks[i].tx = kA;
    }
  }
  L.smem = variant_smem(L.variant, p.num_chunks, (size_t)p.num_stages * p.stage_bytes);
  int64_t total = (int64_t)p.n_tiles * p.tiles_x * p.tiles_y * p.batch;
  int64_t g = (int64_t)kNumSMs * ctas_per_sm;
  if (g > total) g = total;
  g -= g % p.n_tiles;                 // a CTA keeps one N tile's weights resident
  if (g < p.n_tiles) g = p.n_tiles;
  L.grid = (int)g;
}

struct Src {
  const void* base;   // [rows][C] BF16
  int C;              // channels of that buffer
  int c0;             // first channel used
  int nch;            // channels used (multiple of 32)
};

// 1x1 convolution over concatenated sources, flat rows.  BN = 32 or 128.
int build_pointwise(Layer& L, const Src* src, int nsrc, int64_t rows, const void* w_dev, const float* bias_dev,
                    int bn, int act, void* out, int64_t out_pitch, int64_t out_off, int hrb_mask, int lr_h, int lr_w) {
  memset(&L, 0, sizeof(L));
  L.variant = bn == 128 ? V_PW128 : V_PW32;
  IgemmParams& p = L.p;
  int K = 0, nc = 0;
  if (nsrc > kMaxSources) return VSR_ERR_UNSUPPORTED;
  for (int s = 0; s < nsrc; ++s) {
    int rc = make_act_map(&p.a_maps[s], src[s].base, src[s].C, rows, 1, 1, 32, kTileM, 1);
    if (rc) return rc;
    for (int c = 0; c < src[s].nch; c += 32) {
      if (nc >= kMaxChunks) return VSR_ERR_UNSUPPORTED;
      p.chunks[nc].map = (int8_t)s;
      p.chunks[nc].dx = p.chunks[nc].dy = 0;
      p.chunks[nc].c0 = src[s].c0 + c;
      ++nc;
    }
    K += src[s].nch;
  }
  int rc = make_w_map(&p.b_map, w_dev, K, bn, 32, bn);
  if (rc) return rc;
  p.num_chunks = nc;
  p.num_stages = 6;
  p.n_tiles = 1;
  p.tiles_x = (int)ceil_div64(rows, kTileM);
  p.tiles_y = 1;
  p.batch = 1;
  p.tile_w = kTileM;
  p.tile_h = 1;
  p.bias = bias_dev;
  p.bias_n = bn;
  p.act = act;
  p.out = out;
  p.out_pitch = out_pitch;
  p.out_off = out_off;
  p.flat_rows = rows;
  p.lr_h = lr_h;
  p.lr_w = lr_w;
  p.hrb_mask = hrb_mask;
  finish_layer(L, bn == 128 ? 2 : 3);
  const double real_rows = hrb_mask ? (double)rows / ((double)(lr_h + 1) * (lr_w + 1)) * ((double)lr_h * lr_w) : (double)rows;
  L.kclass = bn == 128 ? KC_CONV_IN : (hrb_mask ? KC_PW_HR : KC_PW_LR);
  L.flops = 2.0 * real_rows * K * bn;
  L.bytes = real_rows * (K + bn) * 2.0;
  return VSR_OK;
}

constexpr int kTW = 16, kTH = 8;   // spatial tile (kTW * kTH == 128 rows)

// ConvTranspose2d(32,32,8,4,2): x (B,h,w,32) -> HR block layout (B,h+1,w+1,16,32) or plain NHWC (B,4h,4w,32)
int build_deconv(Layer& L, const void* x, int B, int h, int w, const void* w_dev, const float* bias_dev, void* out,
                 int nhwc) {
  memset(&L, 0, sizeof(L));
  L.variant = V_DECONV;
  IgemmParams& p = L.p;
  // one box per dx: 16 x (8+1) LR pixels; the dy = -1 tap is the box itself, the dy = 0 tap the same box one
  // image row (16 pixels = 1024 bytes, a whole number of swizzle atoms) further in -- 2 TMA boxes per tile, not 4
  int rc = make_act_map(&p.a_maps[0], x, kNF, w, h, B, 32, kTW, kTH + 1);
  if (rc) return rc;
  rc = make_w_map(&p.b_map, w_dev, 4 * kNF, 512, 32, 256);
  if (rc) return rc;
  constexpr int kBox = kTW * (kTH + 1) * 64;   // 9216 bytes
  // chunk t = (dy+1)*2 + (dx+1), tap at LR (Yb+dy, Xb+dx), dy,dx in {-1,0}
  for (int t = 0; t < 4; ++t) {
    const int dyi = t >> 1, dxi = t & 1;
    p.chunks[t].map = 0;
    p.chunks[t].dy = -1;                     // box origin row (both dy taps live in the 9-row box)
    p.chunks[t].dx = (int8_t)(dxi - 1);
    p.chunks[t].c0 = 0;
    p.chunks[t].a_off = dxi * kBox + dyi * (kTW * 64);
    p.chunks[t].tx = dyi == 0 ? kBox : 0;
  }
  p.num_chunks = 4;
  p.cps = 4;            // the 4 taps of a tile share one barrier round trip (the handshake loop of the issuing
  p.stage_bytes = 2 * kBox;   // threads, not the MMAs, was this kernel's floor: ~2000 cycles per tile with one per tap)
  p.num_stages = 4;
  p.n_tiles = 2;
  p.tiles_x = ceil_div(w + 1, kTW);
  p.tiles_y = ceil_div(h + 1, kTH);
  p.batch = B;
  p.tile_w = kTW;
  p.tile_h = kTH;
  p.bias = bias_dev;
  p.bias_n = kNF;
  p.act = 1;
  p.out = out;
  p.lr_h = h;
  p.lr_w = w;
  p.deconv_nhwc = nhwc;
  if (!nhwc) {
    EncodeTiledFn enc = encode_fn();
    if (!enc) return VSR_ERR_STATE;
    cuuint64_t dims[4] = {64, (cuuint64_t)(w + 1), (cuuint64_t)(h + 1), (cuuint64_t)8 * B};
    cuuint64_t strides[3] = {128, (cuuint64_t)128 * (w + 1), (cuuint64_t)128 * (w + 1) * (h + 1)};
    cuuint32_t box[4] = {64, 16, 2, 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(&p.out_map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, out, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return VSR_ERR_CUDA_BASE + 999;
  }
  finish_layer(L, 1);
  const double lrpx = (double)B * h * w;
  L.kclass = KC_DECONV;
  L.flops = lrpx * 131072.0;            // 2 * 64 taps * 32 * 32 per LR pixel
  L.bytes = lrpx * 64.0 * 17.0;         // LR in + 16 HR pixels out, 32 BF16 channels each
  return VSR_OK;
}

// ---- x2 geometry (SRFBN's k6 s2 p2; SURVEY.md 8 a6 / config C4: the reference hard-wires x4) -------------------
// Layered path on plain NHWC HR features: transposed conv (3x3 LR taps, N = 4 sub-positions x 32), 1x1 downtran
// over the concatenated HR maps, strided conv as a 36-tap implicit GEMM.

// ConvTranspose2d(32,32,6,2,2): x (B,h,w,32) -> (B,2h,2w,32) NHWC
int build_deconv2(Layer& L, const void* x, int B, int h, int w, const void* w_dev, const float* bias_dev, void* out) {
  memset(&L, 0, sizeof(L));
  L.variant = V_DECONV2;
  IgemmParams& p = L.p;
  // one 10-row box per dx; the three dy taps are the same box 0 / 1 / 2 image rows (1024 bytes each) further in
  int rc = make_act_map(&p.a_maps[0], x, kNF, w, h, B, 32, kTW, kTH + 2);
  if (rc) return rc;
  rc = make_w_map(&p.b_map, w_dev, 9 * kNF, 128, 32, 128);
  if (rc) return rc;
  {   // output: HR rows of w pixel pairs (128 bytes: rx, channel); one store = 16 pairs of one HR row
    EncodeTiledFn enc = encode_fn();
    if (!enc) return VSR_ERR_STATE;
    cuuint64_t dims[4] = {64, (cuuint64_t)w, (cuuint64_t)2 * h, (cuuint64_t)B};
    cuuint64_t strides[3] = {128, (cuuint64_t)128 * w, (cuuint64_t)256 * w * h};
    cuuint32_t box[4] = {64, (cuuint32_t)kTW, 1, 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(&p.out_map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, out, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return VSR_ERR_CUDA_BASE + 999;
  }
  constexpr int kBox = kTW * (kTH + 2) * 64;   // 10240 bytes
  for (int t = 0; t < 9; ++t) {   // tap at LR (Y+dy, X+dx)
    const int dyi = t / 3, dxi = t % 3;
    p.chunks[t].map = 0;
    p.chunks[t].dy = -1;
    p.chunks[t].dx = (int8_t)(dxi - 1);
    p.chunks[t].c0 = 0;
    p.chunks[t].a_off = dxi * kBox + dyi * (kTW * 64);
    p.chunks[t].tx = dyi == 0 ? kBox : 0;
  }
  p.num_chunks = 9;
  p.cps = 9;
  p.stage_bytes = 3 * kBox;
  p.num_stages = 3;
  p.n_tiles = 1;
  p.tiles_x = ceil_div(w, kTW);
  p.tiles_y = ceil_div(h, kTH);
  p.batch = B;
  p.tile_w = kTW;
  p.tile_h = kTH;
  p.bias = bias_dev;
  p.bias_n = kNF;
  p.act = 1;
  p.out = out;
  p.lr_h = h;
  p.lr_w = w;
  finish_layer(L, 1);
  const double lrpx = (double)B * h * w;
  L.kclass = KC_DECONV;
  L.flops = lrpx * 73728.0;             // 2 * 36 taps * 32 * 32 per LR pixel
  L.bytes = lrpx * 64.0 * 5.0;
  return VSR_OK;
}

// Conv2d(32,32,6,2,2) + PReLU: xhr (B,2h,2w,32) NHWC -> out (B,h,w,32).  Input pixel (2Y-2+ky, 2X-2+kx) with
// (ky, kx) = (2a + py, 2b + px): the row parity py selects one of two tensor maps over every other HR row (no element
// strides); a row of such a map is w pixel pairs of 128 bytes (px, channel) = one K chunk of 64; the three row taps a
// are one 10-row box read 0 / 1 / 2 tile rows (2048 bytes) in; the three column taps b are NOT loaded as shifted boxes:
// they are 3 x 32 accumulator columns (N = 96) and the epilogue adds the neighbours' partials (EPI_DOWN2, 16-column
// tiles that finish their 14 interior columns).  Per 112 output pixels: 2 boxes of 20 KB (1.43 x the HR pixels they
// cover) and 24 MMAs of N = 96, against 12 boxes of 10 KB (3.75 x) and 72 MMAs of N = 32 with the column taps as
// input shifts -- that version kept only 60 KB in flight per SM and ran at the latency of its loads (6.6 ms per
// launch at C4).  TMA zero fill is the padding (column -1 of the first tile included).
int build_downconv2(Layer& L, const void* xhr, int B, int h, int w, const void* w_dev, const float* bias_dev, void* out) {
  memset(&L, 0, sizeof(L));
  L.variant = V_DOWN2;
  IgemmParams& p = L.p;
  EncodeTiledFn enc = encode_fn();
  if (!enc) return VSR_ERR_STATE;
  for (int py = 0; py < 2; ++py) {
    cuuint64_t dims[4] = {64, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)B};
    cuuint64_t strides[3] = {128, (cuuint64_t)256 * w, (cuuint64_t)256 * w * h};
    cuuint32_t box[4] = {64, (cuuint32_t)kTW, (cuuint32_t)kTH + 2, 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    void* base = const_cast<uint8_t*>(reinterpret_cast<const uint8_t*>(xhr)) + (size_t)py * 128 * w;
    CUresult r = enc(&p.a_maps[py], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return VSR_ERR_CUDA_BASE + 999;
  }
  int rc = make_w_map(&p.b_map, w_dev, 6 * 64, 96, 64, 96);
  if (rc) return rc;
  // chunk = py*3 + a (= weight packing order, pack_downconv2); one pipeline stage = one row parity = one box
  constexpr int kBox = kTW * (kTH + 2) * 128;   // 20480 bytes
  for (int py = 0; py < 2; ++py)
    for (int a = 0; a < 3; ++a) {
      Chunk& c = p.chunks[py * 3 + a];
      c.map = (int8_t)py;
      c.dy = -1;
      c.dx = 0;
      c.c0 = 0;
      c.a_off = a * (kTW * 128);
      c.tx = a == 0 ? kBox : 0;
    }
  p.num_chunks = 6;
  p.cps = 3;
  p.stage_bytes = kBox;
  p.num_stages = 6;
  p.n_tiles = 1;
  p.tile_w = kTW - 2;                 // 14 finished columns per 16-column tile
  p.tile_h = kTH;
  p.org_x = -1;
  p.tiles_x = ceil_div(w, kTW - 2);
  p.tiles_y = ceil_div(h, kTH);
  p.batch = B;
  p.bias = bias_dev;
  p.bias_n = kNF;
  p.act = 1;
  p.out = out;
  p.out_pitch = 64;
  p.out_h = h;
  p.out_w = w;
  p.lr_h = h;
  p.lr_w = w;
  finish_layer(L, 1);
  const double lrpx = (double)B * h * w;
  L.kclass = KC_DOWNCONV;
  L.flops = lrpx * 73728.0;
  L.bytes = lrpx * 64.0 * 5.0;
  return VSR_OK;
}

// downtran (1x1 over hr[0..nsrc-1], nsrc >= 2) + PReLU + Conv2d(32,32,8,4,2) pre-activation sums -> acc;
// nsrc == 1: the conv alone on hr[0].  hr[j]: HR block layout (B,h+1,w+1,16,32); acc (B,h,w,32) fp32.
int build_fused_down(Layer& L, const void* const* hr, int nsrc, int B, int h, int w, const void* wt_dev,
                     const float* tran_bias_dev, const void* wd_dev, const float* down_bias_dev, float* part,
                     void* lr_out) {
  memset(&L, 0, sizeof(L));
  const bool tran = nsrc > 1;
  L.variant = tran ? V_FUSED_TRAN : V_FUSED_PLAIN;
  FusedDownParams& f = L.f;
  if (nsrc < 1 || nsrc > kMaxSources) return VSR_ERR_UNSUPPORTED;
  int rc;
  if (tran) {
    for (int j = 0; j < nsrc; ++j) {
      rc = make_act_map(&f.hr_maps[j], hr[j], 64, w + 1, h + 1, 8 * B, 64, 16, 8);   // (el, Xb, Yb, pair plane)
      if (rc) return rc;
    }
    rc = make_w_map(&f.wt_map, wt_dev, 32 * nsrc, 32, 32, 32);
    if (rc) return rc;
  } else {
    rc = make_act_map(&f.h0_map, hr[0], 64, w + 1, h + 1, 8 * B, 64, 16, 8);
    if (rc) return rc;
  }
  rc = make_w_map(&f.wd_map, wd_dev, 512, 128, 64, 128);
  if (rc) return rc;
  f.nsrc = nsrc;
  f.num_stages = tran ? 7 : 5;
  f.tiles_x = ceil_div(w + 1, 16);
  f.tiles_y = ceil_div(h + 1, 8);
  f.batch = B;
  f.lr_h = h;
  f.lr_w = w;
  f.tran_bias = tran_bias_dev;
  f.down_bias = down_bias_dev;
  f.part = part;
  f.lr_out = lr_out;
  // the deepest ring that fits: 4 stages for nsrc 1, 7 for nsrc 2-5, 6 for nsrc 6
  while (f.num_stages > 2 && (tran ? fused_down_smem_bytes<true>(nsrc, f.num_stages)
                                   : fused_down_smem_bytes<false>(nsrc, f.num_stages)) > 227 * 1024)
    --f.num_stages;
  L.smem = tran ? fused_down_smem_bytes<true>(nsrc, f.num_stages) : fused_down_smem_bytes<false>(nsrc, f.num_stages);
  int64_t total = (int64_t)f.tiles_x * f.tiles_y * B;
  L.grid = (int)(total < kNumSMs ? total : kNumSMs);
  const double lrpx = (double)B * h * w;
  L.kclass = KC_FUSED_DOWN;
  L.flops = lrpx * 131072.0 + (tran ? lrpx * 16.0 * 2.0 * 32.0 * nsrc * 32.0 : 0.0);
  L.bytes = lrpx * 64.0 * (16.0 * nsrc) + lrpx * 64.0;   // HR maps in, one BF16 LR map out (slots are not compulsory)
  return VSR_OK;
}

// Feedback groups whose transposed conv runs inside the down kernel (fused_updown_kernel) instead of as its own launch
// in front of it.  The merged kernel does not go below ~2.0 ms per C2 launch (its per-group chain T_U -> U_g -> phase A
// -> H_g -> phase B bounds it, not HBM).  Measured on a B200 at 1000 W against transposed conv + fused down kernel, us
// per launch, nsrc 2..6: 1969 / 1992 / 2002 / 2289 / 2410 against 1762 / 1949 / 2256 / 2657 / 3121 (profiles/
// updown_ab.log).  So groups 3-5 run merged; groups 1-2 and group 0 (no phase A) keep the layered pair.
inline bool updown_merged(int nsrc) { return nsrc >= 4; }

// ConvTranspose2d(32,32,8,4,2) of up_in into hr[nsrc-1] (kept only if `store`) + downtran over hr[0..nsrc-1] + PReLU +
// Conv2d(32,32,8,4,2) pre-activation sums, one launch (fused_updown_kernel); nsrc >= 2.  hr[nsrc-1] may be null when
// !store.
int build_fused_updown(Layer& L, const void* up_in, const void* const* hr, int nsrc, int store, int B, int h, int w,
                       const void* wu_dev, const float* up_bias_dev, const void* wt_dev, const float* tran_bias_dev,
                       const void* wd_dev, const float* down_bias_dev, float* part, void* lr_out) {
  memset(&L, 0, sizeof(L));
  L.variant = V_FUSED_UPDOWN;
  FusedDownParams& f = L.f;
  if (nsrc < 2 || nsrc > kMaxSources || (store && !hr[nsrc - 1])) return VSR_ERR_UNSUPPORTED;
  int rc;
  // hr[0..nsrc-2]: phase-A loads; hr[nsrc-1]: the store view (the same pair-plane boxes)
  for (int j = 0; j < nsrc - (store ? 0 : 1); ++j) {
    rc = make_act_map(&f.hr_maps[j], hr[j], 64, w + 1, h + 1, 8 * B, 64, 16, 8);
    if (rc) return rc;
  }
  rc = make_w_map(&f.wt_map, wt_dev, 32 * nsrc, 32, 32, 32);
  if (rc) return rc;
  rc = make_w_map(&f.wd_map, wd_dev, 512, 128, 64, 128);
  if (rc) return rc;
  rc = make_act_map(&f.up_map, up_in, kNF, w, h, B, 32, kTW, kTH + 1);   // igemm_kernel<EPI_DECONV>'s LR box
  if (rc) return rc;
  rc = make_w_map(&f.wu_map, wu_dev, 4 * kNF, 512, 32, 128);
  if (rc) return rc;
  f.nsrc = nsrc;
  f.tiles_x = ceil_div(w + 1, 16);
  f.tiles_y = ceil_div(h + 1, 8);
  f.batch = B;
  f.lr_h = h;
  f.lr_w = w;
  f.tran_bias = tran_bias_dev;
  f.down_bias = down_bias_dev;
  f.up_bias = up_bias_dev;
  f.part = part;
  f.lr_out = lr_out;
  f.hr_store = store;
  const int64_t total = (int64_t)f.tiles_x * f.tiles_y * B;
  L.grid = (int)(total < kNumSMs ? total : kNumSMs);
  f.num_stages = 7;
  while (f.num_stages > 2 && fused_updown_smem_bytes(nsrc, f.num_stages) > 227 * 1024) --f.num_stages;
  L.smem = fused_updown_smem_bytes(nsrc, f.num_stages);
  const double lrpx = (double)B * h * w;
  L.kclass = KC_FUSED_DOWN;
  L.flops = lrpx * 131072.0 * 2.0 + lrpx * 16.0 * 2.0 * 32.0 * nsrc * 32.0;   // transposed conv + downtran + conv
  // LR map in, nsrc - 1 HR maps in, hr[nsrc-1] out if stored, one BF16 LR map out
  L.bytes = lrpx * 64.0 + lrpx * 64.0 * 16.0 * (nsrc - 1 + (store ? 1 : 0)) + lrpx * 64.0;
  return VSR_OK;
}

int build_finalize(Layer& L, float* acc, const float* bias_dev, void* out, int64_t pixels, int h, int w) {
  memset(&L, 0, sizeof(L));
  L.variant = V_FINALIZE;
  L.fin_acc = acc;
  L.fin_bias = bias_dev;
  L.fin_out = out;
  L.fin_n8 = pixels * 4;
  L.fin_w = w;
  L.fin_h = h;
  L.fin_b = (int)(pixels / ((int64_t)h * w));
  L.kclass = KC_FINALIZE;
  L.flops = 0;
  L.bytes = 0;   // the boundary-pixel pass moves no compulsory bytes (its pixels' output is counted in the fused launch)
  return VSR_OK;
}

// conv_out 3x3 p1 32->3 at HR + bilinear skip + mean shifts, fp32 planar output (B,3,4h,4w)
int build_conv_out(Layer& L, const void* xhr, int B, int h, int w, int scale, const void* w_dev,
                   const float* bias_dev, float* out) {
  memset(&L, 0, sizeof(L));
  L.variant = V_CONVOUT;
  IgemmParams& p = L.p;
  const int H = scale * h, W = scale * w;
  p.inv_scale = 1.0f / (float)scale;
  int rc = make_act_map(&p.a_maps[0], xhr, kNF, W, H, B, 32, 16, 8);
  if (rc) return rc;
  rc = make_w_map(&p.b_map, w_dev, kNF, 32, 32, 32);
  if (rc) return rc;
  p.chunks[0].map = 0;
  p.chunks[0].dx = p.chunks[0].dy = 0;
  p.chunks[0].c0 = 0;
  p.num_chunks = 1;
  p.num_stages = 3;                    // per-tile latency chain (TMEM -> smem exchange -> gather) is hidden by CTAs/SM
  p.n_tiles = 1;
  p.tile_w = 14;                       // 16x8 input tiles produce 14x6 outputs
  p.tile_h = 6;
  p.org_x = -1;
  p.org_y = -1;
  p.tiles_x = ceil_div(W, 14);
  p.tiles_y = ceil_div(H, 6);
  p.batch = B;
  p.bias = bias_dev;
  p.bias_n = 16;
  p.act = 0;
  p.out = out;
  p.out_h = H;
  p.out_w = W;
  p.lr_h = h;
  p.lr_w = w;
  finish_layer(L, 3);
  const double hrpx = (double)B * H * W;
  L.kclass = KC_CONV_OUT;
  L.flops = hrpx * 2.0 * 288 * 3;
  L.bytes = hrpx * (64.0 + 12.0) + hrpx / (scale * scale) * 12.0;
  return VSR_OK;
}

// ------------------------------------------------------------------------------------------------
// weight packing (host): reference state-dict layouts -> K-major BF16 GEMM operands
// ------------------------------------------------------------------------------------------------
inline uint16_t f2bf(float f) {   // round to nearest even, like __float2bfloat16_rn
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

// Conv2d 1x1 weight (N, K, 1, 1) -> [N][K]
void pack_pointwise(const float* w, int N, int K, uint16_t* dst) {
  for (int i = 0; i < N * K; ++i) dst[i] = f2bf(w[i]);
}
// conv_in (128,3,3,3) -> [128][32], k = c*9 + ky*3 + kx, zero padded
void pack_conv_in(const float* w, uint16_t* dst) {
  for (int n = 0; n < 128; ++n)
    for (int k = 0; k < 32; ++k) dst[n * 32 + k] = k < 27 ? f2bf(w[n * 27 + k]) : 0;
}
// ConvTranspose2d weight (c in, o out, 8, 8) -> [512 = s*32+o][128 = t*32+c],
// t = (dy+1)*2+(dx+1), ky = ry - 4*dy, kx = rx - 4*dx   (out y = 4i - 2 + ky)
void pack_deconv(const float* w, uint16_t* dst) {
  for (int s = 0; s < 16; ++s)
    for (int o = 0; o < 32; ++o)
      for (int t = 0; t < 4; ++t)
        for (int c = 0; c < 32; ++c) {
          int ry = s >> 2, rx = s & 3, dy = (t >> 1) - 1, dx = (t & 1) - 1;
          int ky = ry - 4 * dy, kx = rx - 4 * dx;
          dst[(s * 32 + o) * 128 + t * 32 + c] = f2bf(w[((c * 32 + o) * 8 + ky) * 8 + kx]);
        }
}
// Conv2d weight (o, c, 8, 8) s4 p2 for the fused kernel's output-shift form -> [128 = t*32+o][512 = s*32+c],
// tap t = dy*2+dx (block offset of the LR pixel's window), ky = 4dy+ry, kx = 4dx+rx, s = ry*4+rx
void pack_downconv_fused(const float* w, uint16_t* dst) {
  for (int t = 0; t < 4; ++t)
    for (int o = 0; o < 32; ++o)
      for (int s = 0; s < 16; ++s)
        for (int c = 0; c < 32; ++c) {
          int ky = 4 * (t >> 1) + (s >> 2), kx = 4 * (t & 1) + (s & 3);
          dst[(t * 32 + o) * 512 + s * 32 + c] = f2bf(w[((o * 32 + c) * 8 + ky) * 8 + kx]);
        }
}
// x2: ConvTranspose2d weight (c in, o out, 6, 6) s2 p2 -> [128 = s*32+o][288 = t*32+c], s = ry*2+rx,
// t = (dy+1)*3+(dx+1), ky = ry + 2 - 2dy, kx = rx + 2 - 2dx   (out y = 2i - 2 + ky)
void pack_deconv2(const float* w, uint16_t* dst) {
  for (int s = 0; s < 4; ++s)
    for (int o = 0; o < 32; ++o)
      for (int t = 0; t < 9; ++t)
        for (int c = 0; c < 32; ++c) {
          int ry = s >> 1, rx = s & 1, dy = t / 3 - 1, dx = t % 3 - 1;
          int ky = ry + 2 - 2 * dy, kx = rx + 2 - 2 * dx;
          dst[(s * 32 + o) * 288 + t * 32 + c] = f2bf(w[((c * 32 + o) * 6 + ky) * 6 + kx]);
        }
}
// x2: Conv2d weight (o, c, 6, 6) s2 p2 -> [96 = b*32 + o][384 = chunk*64 + px*32 + c], chunk = py*3 + a, for tap
// (ky, kx) = (2a + py, 2b + px) -- the order build_downconv2 issues its K chunks in; the column tap b is an N slice
void pack_downconv2(const float* w, uint16_t* dst) {
  for (int b = 0; b < 3; ++b)
    for (int o = 0; o < 32; ++o)
      for (int py = 0; py < 2; ++py)
        for (int a = 0; a < 3; ++a)
          for (int px = 0; px < 2; ++px) {
            const int chunk = py * 3 + a, ky = 2 * a + py, kx = 2 * b + px;
            for (int c = 0; c < 32; ++c)
              dst[(b * 32 + o) * 384 + chunk * 64 + px * 32 + c] = f2bf(w[((o * 32 + c) * 6 + ky) * 6 + kx]);
          }
}
// conv_out (3,32,3,3) for the output-shift form -> [32 = (ky*3+kx)*3 + o][32 = c], rows 27..31 zero
void pack_conv_out(const float* w, uint16_t* dst) {
  memset(dst, 0, 32 * 32 * 2);
  for (int t = 0; t < 9; ++t)
    for (int o = 0; o < 3; ++o)
      for (int c = 0; c < 32; ++c) dst[(t * 3 + o) * 32 + c] = f2bf(w[(o * 32 + c) * 9 + t]);
}

// ------------------------------------------------------------------------------------------------
// SIMT kernels around the GEMMs
// ------------------------------------------------------------------------------------------------
// sub_mean + zero-padded 3x3 im2col: x (M,3,h,w) f32 -> A0 [M*h*w][32] BF16 (blocks.py:46-55 MeanShift is
// an identity 1x1 conv with bias -255*mean; conv_in pads ITS input, i.e. the shifted image, with zeros).
__global__ void __launch_bounds__(256)
im2col_kernel(const float* __restrict__ x, const float* __restrict__ sub_bias, uint4* __restrict__ a0, int M, int h,
              int w) {
  const int64_t n = (int64_t)M * h * w;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int xx = (int)(i % w), yy = (int)((i / w) % h);
    const int64_t m = i / ((int64_t)h * w);
    float v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = 0.0f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float* pl = x + (m * 3 + c) * (int64_t)h * w;
      const float sb = __ldg(sub_bias + c);
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          int y2 = yy + ky - 1, x2 = xx + kx - 1;
          if (y2 >= 0 && y2 < h && x2 >= 0 && x2 < w) v[c * 9 + ky * 3 + kx] = __ldg(pl + (int64_t)y2 * w + x2) + sb;
        }
    }
    uint4* dst = a0 + i * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      dst[j] = make_uint4(pack_bf16(v[8 * j], v[8 * j + 1]), pack_bf16(v[8 * j + 2], v[8 * j + 3]),
                          pack_bf16(v[8 * j + 4], v[8 * j + 5]), pack_bf16(v[8 * j + 6], v[8 * j + 7]));
  }
}

// fc over the map axis per (channel, HR pixel): Linear(M,32)-ReLU-Linear(32,1)-ReLU
// (SRProjectionModule.py:126-131,146).  maps (W*M,3,H,W) f32 -> y (W,3,H,W) f32: window b = blockIdx.y fuses the
// maps [b*M, (b+1)*M) into frame b with the same per-pixel arithmetic as a one-window launch.
// fcw: [32*M fc0_w][32 fc0_b][32 fc2_w][1 fc2_b]
__global__ void __launch_bounds__(256)
fc_fuse_kernel(const float* __restrict__ maps, const float* __restrict__ fcw, float* __restrict__ y,
               uint8_t* __restrict__ y_u8, int M, int64_t n) {
  maps += (int64_t)blockIdx.y * M * n;
  if (y) y += (int64_t)blockIdx.y * n;
  if (y_u8) y_u8 += (int64_t)blockIdx.y * n;      // the u8 frame (H,W,3) has n bytes
  // y (3,H,W) f32 planar and / or y_u8 (H,W,3): the frame quantised the way the reference's loader stores frames
  // (utils/video_utils.py:23): clamp to 0..255, round half to even -- what a u8 frame writer or gather needs,
  // a quarter of the fp32 bytes.
  __shared__ float s_w[32 * kMaxMaps + 65];
  const int nw = 32 * M + 65;
  for (int i = threadIdx.x; i < nw; i += blockDim.x) s_w[i] = fcw[i];
  __syncthreads();
  const float* w0 = s_w;
  const float* b0 = s_w + 32 * M;
  const float* w2 = b0 + 32;
  const float b2 = w2[32];
  // 4 consecutive outputs per thread: every weight read from shared memory feeds 4 FMAs (with one
  // output per thread the kernel was bound by those LDS, not by the 12 B/pixel/map it streams)
  const int64_t n4 = n >> 2;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += (int64_t)gridDim.x * blockDim.x) {
    float hid[4][32];
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float b = b0[j];
      hid[0][j] = b; hid[1][j] = b; hid[2][j] = b; hid[3][j] = b;
    }
    for (int m0 = 0; m0 < M; m0 += 4) {
      float4 vv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)       // four independent 16-byte loads in flight before the FMAs
        vv[u] = (m0 + u < M) ? ldg_stream_f4(reinterpret_cast<const float4*>(maps + (int64_t)(m0 + u) * n) + q)
                             : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (m0 + u < M) {
          const float4 v = vv[u];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float w = w0[j * M + m0 + u];
            hid[0][j] = fmaf(w, v.x, hid[0][j]);
            hid[1][j] = fmaf(w, v.y, hid[1][j]);
            hid[2][j] = fmaf(w, v.z, hid[2][j]);
            hid[3][j] = fmaf(w, v.w, hid[3][j]);
          }
        }
      }
    }
    float o[4] = {b2, b2, b2, b2};
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float w = w2[j];
#pragma unroll
      for (int k = 0; k < 4; ++k) o[k] = fmaf(w, fmaxf(hid[k][j], 0.0f), o[k]);
    }
    if (y) reinterpret_cast<float4*>(y)[q] = make_float4(fmaxf(o[0], 0.0f), fmaxf(o[1], 0.0f), fmaxf(o[2], 0.0f), fmaxf(o[3], 0.0f));
    if (y_u8) {
      const int64_t hw = n / 3, i0 = q << 2;
      const int64_t c = i0 / hw, p0 = i0 - c * hw;     // hw % 4 == 0 (16 HR pixels per LR pixel): the 4 outputs share c
#pragma unroll
      for (int k = 0; k < 4; ++k) y_u8[(p0 + k) * 3 + c] = (uint8_t)__float2int_rn(fminf(fmaxf(o[k], 0.0f), 255.0f));
    }
  }
  // ragged tail (n is 48*h*w, a multiple of 4 for every LR size; kept for safety)
  for (int64_t i = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float hid[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) hid[j] = b0[j];
    for (int m = 0; m < M; ++m) {
      const float v = __ldg(maps + (int64_t)m * n + i);
#pragma unroll
      for (int j = 0; j < 32; ++j) hid[j] = fmaf(w0[j * M + m], v, hid[j]);
    }
    float o = b2;
#pragma unroll
    for (int j = 0; j < 32; ++j) o = fmaf(w2[j], fmaxf(hid[j], 0.0f), o);
    if (y) y[i] = fmaxf(o, 0.0f);
    if (y_u8) {
      const int64_t hw = n / 3, c = i / hw;
      y_u8[(i - c * hw) * 3 + c] = (uint8_t)__float2int_rn(fminf(fmaxf(o, 0.0f), 255.0f));
    }
  }
}

// Row bands of a stack of `planes` images of `rows` rows (bounds[bands]) x `row` elements each.  Band p holds the rows
// [bounds[p], bounds[p+1]) of every plane, planes one after another (plane stride (bounds[p+1]-bounds[p])*row).  Bands sit
// at band_stride elements apart, or, with band_stride == 0, back to back (band p at bounds[p]*planes*row: the layout of
// the send buffer of an all_to_all with split sizes).
constexpr int kMaxBands = kMaxMaps;
struct BandGeom {
  int bands;
  int bounds[kMaxBands + 1];
  int64_t planes, row, band_stride;
};

// to_bands: image stack -> bands (the exchange's pack); else bands -> image stack (the reorder after a gather).
// blockIdx.y is the band.
template <typename T>
__global__ void __launch_bounds__(256)
band_copy_kernel(const T* __restrict__ src, T* __restrict__ dst, const BandGeom g, int to_bands) {
  const int p = blockIdx.y;
  const int64_t y0 = g.bounds[p], plane_band = (g.bounds[p + 1] - y0) * g.row, plane_img = (int64_t)g.bounds[g.bands] * g.row;
  const int64_t base = g.band_stride ? p * g.band_stride : y0 * g.planes * g.row;
  const int64_t n = g.planes * plane_band;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t k = i / plane_band, r = i - k * plane_band;
    const int64_t img = k * plane_img + y0 * g.row + r;
    if (to_bands) dst[base + i] = __ldg(src + img);
    else dst[img] = __ldg(src + base + i);
  }
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace
}  // namespace vsr

using namespace vsr;

// ------------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------------
enum LayerId : int {
  W_CONV_IN = 0, W_FEAT_IN, W_COMPRESS_IN, W_UPTRAN0, W_UP0 = W_UPTRAN0 + 5, W_DOWNTRAN0 = W_UP0 + 6,
  W_DOWN0 = W_DOWNTRAN0 + 5, W_COMPRESS_OUT = W_DOWN0 + 6, W_OUT, W_CONV_OUT, W_COUNT
};

struct WEntry {
  size_t w_off, b_off;   // byte offsets in the packed buffer
  int N, K;
};

struct vsr_srfbn_plan {
  vsr_srfbn_config cfg;
  WEntry we[W_COUNT];
  size_t fc_off;          // fp32: fc0_w (32*M), fc0_b (32), fc2_w (32), fc2_b (1)
  size_t misc_off;        // fp32: sub_mean bias (3)
  size_t weight_bytes;
  // workspace offsets
  size_t o_a0, o_c128, o_xfeat, o_hidden, o_lr[7], o_u, o_hr[6], o_hb, o_ht, o_acc, o_premix, ws_bytes;
  int chunk_maps;         // maps processed per sweep over the layer list (a divisor of num_maps; == num_maps: no chunking)
  size_t ws_cap;          // caller's workspace cap in bytes (0 = none)
  int windows;            // frame windows per forward: the sweeps run over windows * num_maps maps
  int map0, map1;         // the stack maps this plan sweeps (vsr_srfbn_plan_set_map_range; default [0, num_maps))
  bool bound;
  const uint8_t* dev_w;
  uint8_t* ws;
  std::vector<Layer> layers;
  int conv_out_layer;
  // a second layer list over the maps [refresh_first, num_maps) only (vsr_srfbn_forward_refresh_u8): same buffers,
  // fewer maps; built by vsr_srfbn_prepare_refresh
  std::vector<Layer> refresh_layers;
  int refresh_first, refresh_conv_out_layer;
  bool premix_valid;      // a full forward has filled the per-map images of every map
  std::vector<cudaEvent_t> events;   // profiling: one before every launch + one after the last
  bool profile;
};

static void layout_weights(vsr_srfbn_plan* pl) {
  size_t off = 0;
  auto put = [&](int id, int N, int K, int bias_floats) {
    pl->we[id].N = N;
    pl->we[id].K = K;
    pl->we[id].w_off = off;
    off = align_up(off + (size_t)N * K * 2, 256);
    pl->we[id].b_off = off;
    off = align_up(off + (size_t)bias_floats * 4, 256);
  };
  put(W_CONV_IN, 128, 32, 129);
  put(W_FEAT_IN, 32, 128, 33);
  put(W_COMPRESS_IN, 32, 64, 33);
  for (int i = 0; i < 5; ++i) put(W_UPTRAN0 + i, 32, 32 * (i + 2), 33);
  const bool x2 = pl->cfg.upscale == 2;   // k6 s2 p2: 3x3 LR taps x 4 sub-positions / 36 taps; else k8 s4 p2
  for (int i = 0; i < 6; ++i) put(W_UP0 + i, x2 ? 128 : 512, x2 ? 288 : 128, 33);
  for (int i = 0; i < 5; ++i) put(W_DOWNTRAN0 + i, 32, 32 * (i + 2), 33);
  for (int i = 0; i < 6; ++i) put(W_DOWN0 + i, x2 ? 96 : 128, x2 ? 384 : 512, 33);
  put(W_COMPRESS_OUT, 32, 192, 33);
  put(W_OUT, x2 ? 128 : 512, x2 ? 288 : 128, 33);
  put(W_CONV_OUT, 32, 32, 16 + 7);
  pl->fc_off = off;
  off = align_up(off + (size_t)(32 * pl->cfg.num_maps + 65) * 4, 256);
  pl->misc_off = off;
  off = align_up(off + 16, 256);
  pl->weight_bytes = off;
}

// maps one forward sweeps: all maps of every window, or the plan's map range (one window)
static int swept_maps(const vsr_srfbn_plan* pl) { return pl->windows * (pl->map1 - pl->map0); }

// the plan's range is all maps (no map range set): the only kind of plan that fuses whole frames or has several windows
static bool all_maps(const vsr_srfbn_plan* pl) { return pl->map1 - pl->map0 == pl->cfg.num_maps; }

// Activations are laid out for `chunk` maps at a time (the maps are independent until the fc fuse, so the layer list is
// swept once per chunk); only the per-map SR images in front of the fc fuse exist for all `swept` maps.
static void layout_workspace(vsr_srfbn_plan* pl, int chunk, int swept) {
  const vsr_srfbn_config& c = pl->cfg;
  const size_t P = (size_t)chunk * c.h * c.w;
  const size_t Rb = (size_t)chunk * (c.h + 1) * (c.w + 1) * 16;
  size_t off = 0;
  auto put = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 1024);
    return o;
  };
  pl->o_a0 = put(P * 64);
  pl->o_c128 = put(P * 256);
  pl->o_xfeat = put(P * 64);
  pl->o_hidden = put(P * 64);
  for (int i = 0; i < 7; ++i) pl->o_lr[i] = put(P * 64);
  pl->o_u = put(P * 64);
  const size_t s2 = (size_t)c.upscale * c.upscale;
  const bool x2 = c.upscale == 2;
  // x2: plain NHWC.  x4: hr[5] exists only when its group runs layered (the merged kernel keeps it on chip)
  for (int i = 0; i < 6; ++i) pl->o_hr[i] = put(x2 ? P * s2 * 64 : (i == 5 && updown_merged(6)) ? 0 : Rb * 64);
  pl->o_hb = put(P * s2 * 64);   // plain-NHWC result of the `out` deconv
  pl->o_ht = put(x2 ? P * s2 * 64 : 0);   // x2: downtran result (the x4 path keeps it on chip)
  pl->o_acc = put(x2 ? 0 : P * 512);   // fp32 partial slots of the fused down kernel
  pl->o_premix = put((size_t)swept * c.h * c.w * s2 * 3 * 4);
  pl->ws_bytes = off;
}

// The one place a plan's shape changes: `windows` windows of the maps [m0, m1), in chunks of the largest divisor of
// the swept maps whose workspace fits under ws_cap (no ragged tail chunk: one layer list).  Several windows need the
// range of all maps.  The plan changes only when this returns VSR_OK.
static int set_shape(vsr_srfbn_plan* pl, int windows, int m0, int m1) {
  if (windows > 1 && m1 - m0 != pl->cfg.num_maps) return VSR_ERR_UNSUPPORTED;
  const int swept = windows * (m1 - m0);
  for (int mc = swept; mc >= 1; --mc) {
    if (swept % mc) continue;
    layout_workspace(pl, mc, swept);
    if (pl->ws_cap == 0 || pl->ws_bytes <= pl->ws_cap) {
      pl->windows = windows;
      pl->map0 = m0;
      pl->map1 = m1;
      pl->chunk_maps = mc;
      return VSR_OK;
    }
  }
  layout_workspace(pl, pl->chunk_maps, swept_maps(pl));   // not even one map at a time fits: back to the plan's layout
  return VSR_ERR_WORKSPACE;
}

extern "C" int vsr_srfbn_plan_create(const vsr_srfbn_config* cfg, vsr_srfbn_plan** out_plan) {
  if (!cfg || !out_plan) return VSR_ERR_INVALID_ARG;
  *out_plan = nullptr;
  if (cfg->num_maps < 1 || cfg->h < 1 || cfg->w < 1 || cfg->num_steps < 1) return VSR_ERR_INVALID_ARG;
  // geometry hard-wired by the reference: x4, k8 s4 p2, 32 features, 6 groups (SRProjectionModule.py:97-103);
  // x2 (config C4) uses SRFBN's k6 s2 p2, for which the reference has no code (SURVEY.md 8 a6)
  if (cfg->num_groups != kGroups || cfg->num_features != kNF || (cfg->upscale != 4 && cfg->upscale != 2) ||
      cfg->num_maps > kMaxMaps)
    return VSR_ERR_UNSUPPORTED;
  vsr_srfbn_plan* pl = new (std::nothrow) vsr_srfbn_plan();
  if (!pl) return VSR_ERR_INVALID_ARG;
  pl->cfg = *cfg;
  pl->bound = false;
  pl->dev_w = nullptr;
  pl->ws = nullptr;
  pl->conv_out_layer = -1;
  pl->refresh_first = -1;
  pl->refresh_conv_out_layer = -1;
  pl->premix_valid = false;
  pl->profile = false;
  pl->ws_cap = 0;
  layout_weights(pl);
  set_shape(pl, 1, 0, cfg->num_maps);                  // no cap: always fits unchunked
  *out_plan = pl;
  return VSR_OK;
}

// The cap stays set even when no chunk fits under it, so the setters after it are held to it too.
extern "C" int vsr_srfbn_plan_set_workspace_cap(vsr_srfbn_plan* pl, size_t cap_bytes) {
  if (!pl) return VSR_ERR_INVALID_ARG;
  if (pl->bound) return VSR_ERR_STATE;                // the layer list is built for a chunk size: set the cap before bind
  pl->ws_cap = cap_bytes;
  return set_shape(pl, pl->windows, pl->map0, pl->map1);
}

extern "C" int vsr_srfbn_plan_set_windows(vsr_srfbn_plan* pl, int windows) {
  if (!pl || windows < 1 || windows > 65535) return VSR_ERR_INVALID_ARG;   // fc_fuse_kernel: one grid row per window
  if (pl->bound) return VSR_ERR_STATE;                // buffers and layer list are sized for the window count
  return set_shape(pl, windows, pl->map0, pl->map1);
}

extern "C" int vsr_srfbn_plan_set_map_range(vsr_srfbn_plan* pl, int m0, int m1) {
  if (!pl || m0 < 0 || m1 > pl->cfg.num_maps || m0 >= m1) return VSR_ERR_INVALID_ARG;
  if (pl->bound) return VSR_ERR_STATE;
  if (pl->windows > 1) return VSR_ERR_UNSUPPORTED;     // even the range of all maps
  return set_shape(pl, pl->windows, m0, m1);
}

extern "C" int vsr_srfbn_chunk_maps(const vsr_srfbn_plan* pl) { return pl ? pl->chunk_maps : 0; }

extern "C" void vsr_srfbn_plan_destroy(vsr_srfbn_plan* plan) {
  if (!plan) return;
  for (cudaEvent_t e : plan->events) cudaEventDestroy(e);
  delete plan;
}

extern "C" size_t vsr_srfbn_weight_bytes(const vsr_srfbn_plan* plan) { return plan ? plan->weight_bytes : 0; }
extern "C" size_t vsr_srfbn_workspace_bytes(const vsr_srfbn_plan* plan) { return plan ? plan->ws_bytes : 0; }

extern "C" int vsr_srfbn_pack_weights(const vsr_srfbn_plan* pl, const vsr_srfbn_weights* w, void* host_packed) {
  if (!pl || !w || !host_packed) return VSR_ERR_INVALID_ARG;
  uint8_t* base = reinterpret_cast<uint8_t*>(host_packed);
  memset(base, 0, pl->weight_bytes);
  auto W = [&](int id) { return reinterpret_cast<uint16_t*>(base + pl->we[id].w_off); };
  auto Bv = [&](int id) { return reinterpret_cast<float*>(base + pl->we[id].b_off); };
  auto bias = [&](int id, const float* b, int n, float slope) {
    if (!b) return false;
    memcpy(Bv(id), b, (size_t)n * 4);
    Bv(id)[n] = slope;
    return true;
  };
  bool ok = w->conv_in_w && w->feat_in_w && w->compress_in_w && w->compress_out_w && w->out_w && w->conv_out_w &&
            w->fc0_w && w->fc0_b && w->fc2_w && w->fc2_b && w->sub_mean_bias && w->add_mean_bias;
  for (int i = 0; i < 6; ++i) ok = ok && w->up_w[i] && w->down_w[i];
  for (int i = 0; i < 5; ++i) ok = ok && w->uptran_w[i] && w->downtran_w[i];
  if (!ok) return VSR_ERR_INVALID_ARG;
  pack_conv_in(w->conv_in_w, W(W_CONV_IN));
  ok = ok && bias(W_CONV_IN, w->conv_in_b, 128, w->conv_in_slope);
  pack_pointwise(w->feat_in_w, 32, 128, W(W_FEAT_IN));
  ok = ok && bias(W_FEAT_IN, w->feat_in_b, 32, w->feat_in_slope);
  pack_pointwise(w->compress_in_w, 32, 64, W(W_COMPRESS_IN));
  ok = ok && bias(W_COMPRESS_IN, w->compress_in_b, 32, w->compress_in_slope);
  for (int i = 0; i < 5; ++i) {
    pack_pointwise(w->uptran_w[i], 32, 32 * (i + 2), W(W_UPTRAN0 + i));
    ok = ok && bias(W_UPTRAN0 + i, w->uptran_b[i], 32, w->uptran_slope[i]);
    pack_pointwise(w->downtran_w[i], 32, 32 * (i + 2), W(W_DOWNTRAN0 + i));
    ok = ok && bias(W_DOWNTRAN0 + i, w->downtran_b[i], 32, w->downtran_slope[i]);
  }
  const bool x2 = pl->cfg.upscale == 2;
  for (int i = 0; i < 6; ++i) {
    if (x2) pack_deconv2(w->up_w[i], W(W_UP0 + i));
    else pack_deconv(w->up_w[i], W(W_UP0 + i));
    ok = ok && bias(W_UP0 + i, w->up_b[i], 32, w->up_slope[i]);
    if (x2) pack_downconv2(w->down_w[i], W(W_DOWN0 + i));
    else pack_downconv_fused(w->down_w[i], W(W_DOWN0 + i));
    ok = ok && bias(W_DOWN0 + i, w->down_b[i], 32, w->down_slope[i]);
  }
  pack_pointwise(w->compress_out_w, 32, 192, W(W_COMPRESS_OUT));
  ok = ok && bias(W_COMPRESS_OUT, w->compress_out_b, 32, w->compress_out_slope);
  if (x2) pack_deconv2(w->out_w, W(W_OUT));
  else pack_deconv(w->out_w, W(W_OUT));
  ok = ok && bias(W_OUT, w->out_b, 32, w->out_slope);
  pack_conv_out(w->conv_out_w, W(W_CONV_OUT));
  if (!w->conv_out_b) return VSR_ERR_INVALID_ARG;
  {
    float* b = Bv(W_CONV_OUT);
    memcpy(b, w->conv_out_b, 3 * 4);
    b[16] = 0.0f;
    memcpy(b + 17, w->sub_mean_bias, 3 * 4);
    memcpy(b + 20, w->add_mean_bias, 3 * 4);
  }
  if (!ok) return VSR_ERR_INVALID_ARG;
  const int M = pl->cfg.num_maps;
  float* fc = reinterpret_cast<float*>(base + pl->fc_off);
  memcpy(fc, w->fc0_w, (size_t)32 * M * 4);
  memcpy(fc + 32 * M, w->fc0_b, 32 * 4);
  memcpy(fc + 32 * M + 32, w->fc2_w, 32 * 4);
  fc[32 * M + 64] = w->fc2_b[0];
  memcpy(base + pl->misc_off, w->sub_mean_bias, 3 * 4);
  return VSR_OK;
}

static int build_layer_list(vsr_srfbn_plan* pl, int M, std::vector<Layer>& layers, int& conv_out_layer);

extern "C" int vsr_srfbn_bind(vsr_srfbn_plan* pl, const void* dev_weights, void* dev_workspace,
                              size_t workspace_bytes) {
  if (!pl || !dev_weights || !dev_workspace) return VSR_ERR_INVALID_ARG;
  if (workspace_bytes < pl->ws_bytes) return VSR_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(dev_weights) % 256 || reinterpret_cast<uintptr_t>(dev_workspace) % 256)
    return VSR_ERR_INVALID_ARG;
  pl->bound = false;
  pl->dev_w = reinterpret_cast<const uint8_t*>(dev_weights);
  pl->ws = reinterpret_cast<uint8_t*>(dev_workspace);
  pl->refresh_layers.clear();
  pl->refresh_first = -1;
  pl->premix_valid = false;
  int rc = build_layer_list(pl, pl->chunk_maps, pl->layers, pl->conv_out_layer);
  if (rc) return rc;
  pl->bound = true;
  return VSR_OK;
}

// The layer list of the stack for M maps at a time (M <= chunk_maps: the buffers are laid out for chunk_maps maps and a
// list over fewer maps uses their heads).
static int build_layer_list(vsr_srfbn_plan* pl, int M, std::vector<Layer>& layers, int& conv_out_layer) {
  layers.clear();
  const vsr_srfbn_config& c = pl->cfg;
  const int h = c.h, w = c.w;
  const int64_t P = (int64_t)M * h * w;
  uint8_t* ws = pl->ws;
  auto Wp = [&](int id) { return (const void*)(pl->dev_w + pl->we[id].w_off); };
  auto Bp = [&](int id) { return reinterpret_cast<const float*>(pl->dev_w + pl->we[id].b_off); };
  int rc;
  Layer L;
#define PUSH(expr)        \
  do {                    \
    rc = (expr);          \
    if (rc) return rc;    \
    layers.push_back(L);  \
  } while (0)

  {  // conv_in: A0 [P,32] -> C128 [P,128]
    Src s{ws + pl->o_a0, 32, 0, 32};
    PUSH(build_pointwise(L, &s, 1, P, Wp(W_CONV_IN), Bp(W_CONV_IN), 128, 1, ws + pl->o_c128, 256, 0, 0, h, w));
  }
  {  // feat_in: C128 -> xfeat
    Src s{ws + pl->o_c128, 128, 0, 128};
    PUSH(build_pointwise(L, &s, 1, P, Wp(W_FEAT_IN), Bp(W_FEAT_IN), 32, 1, ws + pl->o_xfeat, 64, 0, 0, h, w));
  }
  for (int step = 0; step < c.num_steps; ++step) {
    {  // compress_in(cat(x, last_hidden)); first step: last_hidden = x (SRProjectionModule.py:45-48)
      Src s[2] = {{ws + pl->o_xfeat, 32, 0, 32}, {ws + (step == 0 ? pl->o_xfeat : pl->o_hidden), 32, 0, 32}};
      PUSH(build_pointwise(L, s, 2, P, Wp(W_COMPRESS_IN), Bp(W_COMPRESS_IN), 32, 1, ws + pl->o_lr[0], 64, 0, 0, h, w));
    }
    for (int i = 0; i < kGroups; ++i) {
      const void* up_in = ws + pl->o_lr[0];
      if (i > 0) {  // uptran(cat(lr[0..i]))
        Src s[6];
        for (int j = 0; j <= i; ++j) s[j] = Src{ws + pl->o_lr[j], 32, 0, 32};
        PUSH(build_pointwise(L, s, i + 1, P, Wp(W_UPTRAN0 + i - 1), Bp(W_UPTRAN0 + i - 1), 32, 1, ws + pl->o_u, 64, 0,
                             0, h, w));
        up_in = ws + pl->o_u;
      }
      if (c.upscale == 2) {
        PUSH(build_deconv2(L, up_in, M, h, w, Wp(W_UP0 + i), Bp(W_UP0 + i), ws + pl->o_hr[i]));
        const void* down_in = ws + pl->o_hr[0];
        if (i > 0) {  // downtran(cat(hr[0..i])) over flat HR rows
          Src s[6];
          for (int j = 0; j <= i; ++j) s[j] = Src{ws + pl->o_hr[j], 32, 0, 32};
          rc = build_pointwise(L, s, i + 1, P * 4, Wp(W_DOWNTRAN0 + i - 1), Bp(W_DOWNTRAN0 + i - 1), 32, 1,
                               ws + pl->o_ht, 64, 0, 0, h, w);
          if (rc) return rc;
          L.kclass = KC_PW_HR;
          layers.push_back(L);
          down_in = ws + pl->o_ht;
        }
        PUSH(build_downconv2(L, down_in, M, h, w, Wp(W_DOWN0 + i), Bp(W_DOWN0 + i), ws + pl->o_lr[i + 1]));
        continue;
      }
      if (updown_merged(i + 1)) {   // upBlocks[i] + downtran(cat(hr[0..i])) + downBlocks[i] in one launch
        const void* hrs[6];
        for (int j = 0; j <= i; ++j) hrs[j] = ws + pl->o_hr[j];
        const int store = i + 1 < kGroups;     // hr[5] is read by no later group
        if (!store) hrs[i] = nullptr;
        PUSH(build_fused_updown(L, up_in, hrs, i + 1, store, M, h, w, Wp(W_UP0 + i), Bp(W_UP0 + i),
                                Wp(W_DOWNTRAN0 + i - 1), Bp(W_DOWNTRAN0 + i - 1), Wp(W_DOWN0 + i), Bp(W_DOWN0 + i),
                                reinterpret_cast<float*>(ws + pl->o_acc), ws + pl->o_lr[i + 1]));
        PUSH(build_finalize(L, reinterpret_cast<float*>(ws + pl->o_acc), Bp(W_DOWN0 + i), ws + pl->o_lr[i + 1], P, h, w));
      } else {  // upBlocks[i], then downtran(cat(hr[0..i])) + downBlocks[i] fused; sums land in the fp32 LR accumulator
        Layer D, F;
        rc = build_deconv(D, up_in, M, h, w, Wp(W_UP0 + i), Bp(W_UP0 + i), ws + pl->o_hr[i], 0);
        if (rc) return rc;
        const void* hrs[6];
        for (int j = 0; j <= i; ++j) hrs[j] = ws + pl->o_hr[j];
        rc = build_fused_down(F, hrs, i + 1, M, h, w, i > 0 ? Wp(W_DOWNTRAN0 + i - 1) : nullptr,
                              i > 0 ? Bp(W_DOWNTRAN0 + i - 1) : nullptr, Wp(W_DOWN0 + i), Bp(W_DOWN0 + i),
                              reinterpret_cast<float*>(ws + pl->o_acc), ws + pl->o_lr[i + 1]);
        if (rc) return rc;
        layers.push_back(D);
        layers.push_back(F);
        PUSH(build_finalize(L, reinterpret_cast<float*>(ws + pl->o_acc), Bp(W_DOWN0 + i), ws + pl->o_lr[i + 1], P, h, w));
      }
    }
    {  // compress_out(cat(lr[1..6])) -> hidden
      Src s[6];
      for (int j = 0; j < 6; ++j) s[j] = Src{ws + pl->o_lr[j + 1], 32, 0, 32};
      PUSH(build_pointwise(L, s, 6, P, Wp(W_COMPRESS_OUT), Bp(W_COMPRESS_OUT), 32, 1, ws + pl->o_hidden, 64, 0, 0, h,
                           w));
    }
  }
  if (c.upscale == 2) PUSH(build_deconv2(L, ws + pl->o_hidden, M, h, w, Wp(W_OUT), Bp(W_OUT), ws + pl->o_hb));
  else PUSH(build_deconv(L, ws + pl->o_hidden, M, h, w, Wp(W_OUT), Bp(W_OUT), ws + pl->o_hb, 1));
  PUSH(build_conv_out(L, ws + pl->o_hb, M, h, w, c.upscale, Wp(W_CONV_OUT), Bp(W_CONV_OUT),
                      reinterpret_cast<float*>(ws + pl->o_premix)));
  conv_out_layer = (int)layers.size() - 1;
#undef PUSH
  return VSR_OK;
}

// Prepares vsr_srfbn_forward_refresh_u8 / vsr_srfbn_forward_maps_refresh for the maps [first_map, num_maps), of which a
// plan with a map range sweeps [max(first_map, map0), map1) -- possibly none.
extern "C" int vsr_srfbn_prepare_refresh(vsr_srfbn_plan* pl, int first_map) {
  if (!pl) return VSR_ERR_INVALID_ARG;
  if (!pl->bound) return VSR_ERR_STATE;
  if (first_map < 1 || first_map >= pl->cfg.num_maps) return VSR_ERR_INVALID_ARG;
  if (pl->chunk_maps != swept_maps(pl)) return VSR_ERR_UNSUPPORTED;   // not with chunked sweeps
  if (pl->refresh_first == first_map) return VSR_OK;
  pl->refresh_first = -1;
  pl->refresh_layers.clear();
  const int count = pl->map1 - std::max(first_map, pl->map0);
  if (count > 0) {
    const int rc = build_layer_list(pl, count, pl->refresh_layers, pl->refresh_conv_out_layer);
    if (rc) return rc;
  }
  pl->refresh_first = first_map;
  return VSR_OK;
}

extern "C" int vsr_srfbn_forward(vsr_srfbn_plan* pl, const float* x, float* y, vsr_stream_t stream) {
  return vsr_srfbn_forward_u8(pl, x, y, nullptr, stream);
}

// One sweep of a layer list over the maps [m0, m0 + Mc) of the stack x; the per-map image of map m lands in premix slot
// m - map0 (several windows imply map0 == 0, so window b's map m lands in slot b*M + m).
static int sweep_maps(vsr_srfbn_plan* pl, std::vector<Layer>& layers, int conv_out_layer, const float* x, int m0, int Mc,
                      cudaStream_t st, size_t* ev) {
  const vsr_srfbn_config& c = pl->cfg;
  const int64_t P = (int64_t)Mc * c.h * c.w;
  auto mark = [&]() {
    if (ev && pl->profile && *ev < pl->events.size()) cudaEventRecord(pl->events[(*ev)++], st);
  };
  const float* xc = x + (int64_t)m0 * 3 * c.h * c.w;
  mark();
  {
    int64_t blocks = ceil_div64(P, 256);
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    im2col_kernel<<<(int)blocks, 256, 0, st>>>(xc, reinterpret_cast<const float*>(pl->dev_w + pl->misc_off),
                                               reinterpret_cast<uint4*>(pl->ws + pl->o_a0), Mc, c.h, c.w);
    int rc = after_launch();
    if (rc) return rc;
  }
  {   // the last layer reads the network input (bilinear skip) and writes these maps of the premix buffer
    IgemmParams& cp = layers[conv_out_layer].p;
    cp.skip_src = xc;
    cp.out = reinterpret_cast<float*>(pl->ws + pl->o_premix) + (int64_t)(m0 - pl->map0) * 3 * c.upscale * c.upscale * c.h * c.w;
  }
  for (const Layer& L : layers) {
    mark();
    int rc = launch_layer(L, st);
    if (rc) return rc;
  }
  return VSR_OK;
}

// The full forward's sweeps: the plan's maps [map0, map0 + swept_maps) in chunks of chunk_maps.
static int sweep_all(vsr_srfbn_plan* pl, const float* x, cudaStream_t st, size_t* ev) {
  for (int m0 = pl->map0; m0 < pl->map0 + swept_maps(pl); m0 += pl->chunk_maps) {
    int rc = sweep_maps(pl, pl->layers, pl->conv_out_layer, x, m0, pl->chunk_maps, st, ev);
    if (rc) return rc;
  }
  return VSR_OK;
}

// The refresh forward's sweeps: the maps of window b that changed since the last forward and lie in the plan's range,
// [b*M + max(first_map, map0), b*M + map1), one sweep of the refresh layer list per window -- none when that range is
// empty.  The stack keeps the caller's window-major layout, so no map is copied or reordered to make the changed maps
// of all windows contiguous; the price is windows sweeps instead of one, which only matters where launches dominate.
static int sweep_changed(vsr_srfbn_plan* pl, int first_map, const float* x, cudaStream_t st) {
  const int M = pl->cfg.num_maps, m0 = std::max(first_map, pl->map0);
  if (m0 >= pl->map1) return VSR_OK;
  for (int b = 0; b < pl->windows; ++b) {
    int rc = sweep_maps(pl, pl->refresh_layers, pl->refresh_conv_out_layer, x, b * M + m0, pl->map1 - m0, st, nullptr);
    if (rc) return rc;
  }
  return VSR_OK;
}

// the per-pixel fc across num_maps images of n floats each (maps (windows*num_maps, n)), one window per grid row
static int launch_fc(vsr_srfbn_plan* pl, const float* maps, float* y, uint8_t* y_u8, int64_t n, int windows,
                     cudaStream_t st) {
  int64_t blocks = ceil_div64(ceil_div64(n, 4), 256);
  if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
  fc_fuse_kernel<<<dim3((unsigned)blocks, (unsigned)windows), 256, 0, st>>>(
      maps, reinterpret_cast<const float*>(pl->dev_w + pl->fc_off), y, y_u8, pl->cfg.num_maps, n);
  return after_launch();
}

// the per-pixel fc across the num_maps per-map images of each window (SRProjectionModule.py:146), one window per grid row
static int fuse_maps(vsr_srfbn_plan* pl, float* y, uint8_t* y_u8, cudaStream_t st) {
  const vsr_srfbn_config& c = pl->cfg;
  const int64_t n = (int64_t)3 * c.upscale * c.upscale * c.h * c.w;
  return launch_fc(pl, reinterpret_cast<const float*>(pl->ws + pl->o_premix), y, y_u8, n, pl->windows, st);
}

extern "C" int vsr_srfbn_forward_u8(vsr_srfbn_plan* pl, const float* x, float* y, uint8_t* y_u8, vsr_stream_t stream) {
  if (!pl || !x || (!y && !y_u8)) return VSR_ERR_INVALID_ARG;
  if (!pl->bound) return VSR_ERR_STATE;
  if (!all_maps(pl)) return VSR_ERR_UNSUPPORTED;      // a map range fuses by bands
  cudaStream_t st = as_stream(stream);
  size_t ev = 0;
  int rc = sweep_all(pl, x, st, &ev);
  if (rc) return rc;
  if (pl->profile && ev < pl->events.size()) cudaEventRecord(pl->events[ev++], st);
  rc = fuse_maps(pl, y, y_u8, st);
  if (rc) return rc;
  if (pl->profile && ev < pl->events.size()) cudaEventRecord(pl->events[ev++], st);
  pl->premix_valid = true;
  return VSR_OK;
}

// A second call on a stack of which only the maps [first_map, num_maps) changed since the last forward of this plan
// (the fuse pass of network/video_super_resolution.py:62: `data`, the frames, goes in unchanged): the maps are
// independent until the per-pixel fc, so the per-map images of the unchanged maps are still in the workspace and only
// the changed ones are swept again -- bit-identical to a full forward on the same stack.  Needs
// vsr_srfbn_prepare_refresh(plan, first_map) and a preceding vsr_srfbn_forward[_u8] on the same stream.
extern "C" int vsr_srfbn_forward_refresh_u8(vsr_srfbn_plan* pl, const float* x, float* y, uint8_t* y_u8, int first_map,
                                            vsr_stream_t stream) {
  if (!pl || !x || (!y && !y_u8)) return VSR_ERR_INVALID_ARG;
  if (!pl->bound || !pl->premix_valid || pl->refresh_first != first_map || first_map < 1) return VSR_ERR_STATE;
  if (!all_maps(pl)) return VSR_ERR_UNSUPPORTED;
  cudaStream_t st = as_stream(stream);
  int rc = sweep_changed(pl, first_map, x, st);
  if (rc) return rc;
  return fuse_maps(pl, y, y_u8, st);
}

// ---- map-parallel forward: the plan's map range, row bands, band fuse ----

extern "C" int vsr_srfbn_forward_maps(vsr_srfbn_plan* pl, const float* x, vsr_stream_t stream) {
  if (!pl || !x) return VSR_ERR_INVALID_ARG;
  if (!pl->bound) return VSR_ERR_STATE;
  int rc = sweep_all(pl, x, as_stream(stream), nullptr);
  if (rc) return rc;
  pl->premix_valid = true;
  return VSR_OK;
}

extern "C" int vsr_srfbn_forward_maps_refresh(vsr_srfbn_plan* pl, const float* x, int first_map, vsr_stream_t stream) {
  if (!pl || !x) return VSR_ERR_INVALID_ARG;
  if (!pl->bound || !pl->premix_valid || pl->refresh_first != first_map || first_map < 1) return VSR_ERR_STATE;
  if (pl->windows > 1) return VSR_ERR_UNSUPPORTED;
  return sweep_changed(pl, first_map, x, as_stream(stream));
}

// bounds[0] == 0 < bounds[1] < ... < bounds[bands] == total, 1 <= bands <= kMaxBands
static bool bands_ok(const int* bounds, int bands, int total) {
  if (!bounds || bands < 1 || bands > kMaxBands || bounds[0] != 0 || bounds[bands] != total) return false;
  for (int p = 0; p < bands; ++p)
    if (bounds[p + 1] <= bounds[p]) return false;
  return true;
}

static int launch_band_copy(const void* src, void* dst, int elem_bytes, const BandGeom& g, int to_bands,
                            cudaStream_t st) {
  int max_rows = 0;
  for (int p = 0; p < g.bands; ++p) max_rows = std::max(max_rows, g.bounds[p + 1] - g.bounds[p]);
  int64_t blocks = ceil_div64(g.planes * max_rows * g.row, 256);
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  const dim3 grid((unsigned)blocks, (unsigned)g.bands);
  if (elem_bytes == 4)
    band_copy_kernel<uint32_t><<<grid, 256, 0, st>>>(reinterpret_cast<const uint32_t*>(src),
                                                     reinterpret_cast<uint32_t*>(dst), g, to_bands);
  else
    band_copy_kernel<uint8_t><<<grid, 256, 0, st>>>(reinterpret_cast<const uint8_t*>(src),
                                                    reinterpret_cast<uint8_t*>(dst), g, to_bands);
  return after_launch();
}

extern "C" int vsr_srfbn_pack_bands(const vsr_srfbn_plan* pl, const int* lr_bounds, int bands, float* send,
                                    vsr_stream_t stream) {
  if (!pl || !send || !bands_ok(lr_bounds, bands, pl->cfg.h)) return VSR_ERR_INVALID_ARG;
  if (!pl->bound) return VSR_ERR_STATE;
  if (pl->windows > 1) return VSR_ERR_UNSUPPORTED;
  const vsr_srfbn_config& c = pl->cfg;
  BandGeom g;
  g.bands = bands;
  for (int p = 0; p <= bands; ++p) g.bounds[p] = lr_bounds[p] * c.upscale;
  g.planes = (int64_t)(pl->map1 - pl->map0) * 3;
  g.row = (int64_t)c.upscale * c.w;
  g.band_stride = 0;
  return launch_band_copy(pl->ws + pl->o_premix, send, 4, g, 1, as_stream(stream));
}

extern "C" int vsr_srfbn_fuse_band(vsr_srfbn_plan* pl, const float* maps, int rows, float* y_band, uint8_t* y_u8_band,
                                   vsr_stream_t stream) {
  if (!pl || !maps || (!y_band && !y_u8_band)) return VSR_ERR_INVALID_ARG;
  if (!pl->bound) return VSR_ERR_STATE;
  const vsr_srfbn_config& c = pl->cfg;
  // whole LR rows: every map plane of the band is a multiple of 16 bytes and 4 consecutive outputs share a channel
  if (rows < 1 || rows % c.upscale || rows > c.upscale * c.h) return VSR_ERR_INVALID_ARG;
  if (reinterpret_cast<uintptr_t>(maps) % 16 || reinterpret_cast<uintptr_t>(y_band) % 16) return VSR_ERR_INVALID_ARG;
  return launch_fc(pl, maps, y_band, y_u8_band, (int64_t)3 * rows * c.upscale * c.w, 1, as_stream(stream));
}

extern "C" int vsr_unpack_bands(const void* bands_src, void* dst, int elem_bytes, int64_t planes, int64_t row,
                                const int* bounds, int bands, int64_t band_stride, vsr_stream_t stream) {
  if (!bands_src || !dst || (elem_bytes != 1 && elem_bytes != 4) || planes < 1 || row < 1 || band_stride < 0 ||
      !bounds || bands < 1 || bands > kMaxBands || !bands_ok(bounds, bands, bounds[bands]))
    return VSR_ERR_INVALID_ARG;
  if (elem_bytes == 4 && (reinterpret_cast<uintptr_t>(bands_src) % 4 || reinterpret_cast<uintptr_t>(dst) % 4))
    return VSR_ERR_INVALID_ARG;
  BandGeom g;
  g.bands = bands;
  for (int p = 0; p <= bands; ++p) {
    g.bounds[p] = bounds[p];
    if (p < bands && band_stride && planes * (bounds[p + 1] - bounds[p]) * row > band_stride) return VSR_ERR_INVALID_ARG;
  }
  g.planes = planes;
  g.row = row;
  g.band_stride = band_stride;
  return launch_band_copy(bands_src, dst, elem_bytes, g, 0, as_stream(stream));
}

extern "C" const char* vsr_srfbn_kernel_class_name(int k) {
  static const char* names[KC_COUNT] = {"im2col", "conv_in_gemm", "pointwise_lr", "pointwise_hr", "deconv8x8s4",
                                        "conv8x8s4", "conv_out3x3", "fc_fuse", "fused_downtran_conv8x8s4",
                                        "finalize_lr"};
  return (k >= 0 && k < KC_COUNT) ? names[k] : "?";
}

extern "C" int vsr_srfbn_profile_enable(vsr_srfbn_plan* pl, int enable) {
  if (!pl) return VSR_ERR_INVALID_ARG;
  if (!pl->bound) return VSR_ERR_STATE;
  pl->profile = enable != 0;
  if (pl->profile && pl->events.empty()) {
    pl->events.resize((pl->layers.size() + 1) * (size_t)(swept_maps(pl) / pl->chunk_maps) + 2);
    for (cudaEvent_t& e : pl->events) {
      cudaError_t r = cudaEventCreate(&e);
      if (r != cudaSuccess) return cuda_status(r);
    }
  }
  return VSR_OK;
}

struct ProfiledLaunch {
  int kclass;
  double flops, bytes;
};

// The launch between events i and i + 1 of a profiled vsr_srfbn_forward_u8: per chunk sweep an im2col and the layer
// list, then the fc fuse in the last interval.
static ProfiledLaunch profiled_launch(const vsr_srfbn_plan* pl, size_t i) {
  const vsr_srfbn_config& c = pl->cfg;
  const size_t per = pl->layers.size() + 1;   // launches per chunk sweep
  if (i == pl->events.size() - 2) {
    const double s2 = (double)c.upscale * c.upscale, Pall = (double)pl->windows * c.num_maps * c.h * c.w;
    return {KC_FC, s2 * Pall / c.num_maps * 3 * 2.0 * (32.0 * c.num_maps + 32.0),
            s2 * Pall * 12.0 + s2 * Pall / c.num_maps * 12.0};
  }
  if (i % per == 0) return {KC_IM2COL, 0, (double)pl->chunk_maps * c.h * c.w * (12.0 + 64.0)};
  const Layer& L = pl->layers[i % per - 1];
  return {L.kclass, L.flops, L.bytes};
}

extern "C" int vsr_srfbn_profile_read(vsr_srfbn_plan* pl, double* ms, int32_t* launches, double* flops, double* bytes) {
  if (!pl || !ms || !launches || !flops || !bytes) return VSR_ERR_INVALID_ARG;
  if (!pl->bound || pl->events.empty()) return VSR_ERR_STATE;
  for (int k = 0; k < VSR_SRFBN_KERNEL_CLASSES; ++k) { ms[k] = 0; launches[k] = 0; flops[k] = 0; bytes[k] = 0; }
  cudaError_t r = cudaEventSynchronize(pl->events.back());
  if (r != cudaSuccess) return cuda_status(r);
  for (size_t i = 0; i + 1 < pl->events.size(); ++i) {
    float t = 0;
    r = cudaEventElapsedTime(&t, pl->events[i], pl->events[i + 1]);
    if (r != cudaSuccess) return cuda_status(r);
    const ProfiledLaunch l = profiled_launch(pl, i);
    ms[l.kclass] += t; launches[l.kclass] += 1; flops[l.kclass] += l.flops; bytes[l.kclass] += l.bytes;
  }
  return VSR_OK;
}

extern "C" int vsr_srfbn_profile_launches(vsr_srfbn_plan* pl, float* ms, int32_t* kclass, int32_t capacity) {
  if (!pl || !ms || !kclass) return -1;
  if (!pl->bound || pl->events.empty()) return -1;
  if (cudaEventSynchronize(pl->events.back()) != cudaSuccess) return -1;
  const size_t n = pl->events.size() - 1;
  for (size_t i = 0; i < n && (int32_t)i < capacity; ++i) {
    float t = 0;
    cudaEventElapsedTime(&t, pl->events[i], pl->events[i + 1]);
    ms[i] = t;
    kclass[i] = profiled_launch(pl, i).kclass;
  }
  return (int)n;
}

extern "C" int vsr_srfbn_debug_premix(const vsr_srfbn_plan* pl, float* out_maps, vsr_stream_t stream) {
  if (!pl || !out_maps) return VSR_ERR_INVALID_ARG;
  if (!pl->bound) return VSR_ERR_STATE;
  const vsr_srfbn_config& c = pl->cfg;
  size_t bytes = (size_t)swept_maps(pl) * 3 * c.upscale * c.upscale * c.h * c.w * 4;
  return cuda_status(cudaMemcpyAsync(out_maps, pl->ws + pl->o_premix, bytes, cudaMemcpyDeviceToDevice, as_stream(stream)));
}

// ------------------------------------------------------------------------------------------------
// single-layer test hooks: same kernels, same packing, one layer
// ------------------------------------------------------------------------------------------------
extern "C" size_t vsr_test_workspace_bytes(int B, int h, int w) {
  (void)B; (void)h; (void)w;
  return 512 * 1024;   // packed weights (<= 128 KB) + bias
}

static int upload(void* dev, const void* host, size_t bytes, cudaStream_t st) {
  cudaError_t e = cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) return cuda_status(e);
  return cuda_status(cudaStreamSynchronize(st));   // the host staging vector dies with the caller
}

extern "C" int vsr_test_pointwise(const void* x_bf16, int64_t rows, int K, const float* w_host, const float* b_host,
                                  float slope, int act, void* y_bf16, void* workspace, size_t workspace_bytes,
                                  vsr_stream_t stream) {
  if (!x_bf16 || !w_host || !b_host || !y_bf16 || !workspace || rows <= 0) return VSR_ERR_INVALID_ARG;
  if (K % 32 || K < 32 || K > 224) return VSR_ERR_UNSUPPORTED;
  if (workspace_bytes < vsr_test_workspace_bytes(1, 1, 1)) return VSR_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  std::vector<uint16_t> wp((size_t)32 * K);
  pack_pointwise(w_host, 32, K, wp.data());
  float bias[33];
  memcpy(bias, b_host, 32 * 4);
  bias[32] = slope;
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  int rc = upload(ws, wp.data(), wp.size() * 2, st);
  if (rc) return rc;
  rc = upload(ws + 256 * 1024, bias, sizeof(bias), st);
  if (rc) return rc;
  Layer L;
  Src s{x_bf16, K, 0, K};
  rc = build_pointwise(L, &s, 1, rows, ws, reinterpret_cast<const float*>(ws + 256 * 1024), 32, act, y_bf16, 64, 0, 0,
                       1, 1);
  if (rc) return rc;
  rc = launch_layer(L, st);
  if (rc) return rc;
  return cuda_status(cudaStreamSynchronize(st));
}

extern "C" int vsr_test_deconv(const void* x_bf16, int B, int h, int w, const float* w_host, const float* b_host,
                               float slope, int block_layout, void* y_bf16, void* workspace,
                               size_t workspace_bytes, vsr_stream_t stream) {
  if (!x_bf16 || !w_host || !b_host || !y_bf16 || !workspace || B <= 0 || h <= 0 || w <= 0) return VSR_ERR_INVALID_ARG;
  if (workspace_bytes < vsr_test_workspace_bytes(B, h, w)) return VSR_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  std::vector<uint16_t> wp((size_t)512 * 128);
  pack_deconv(w_host, wp.data());
  float bias[33];
  memcpy(bias, b_host, 32 * 4);
  bias[32] = slope;
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  int rc = upload(ws, wp.data(), wp.size() * 2, st);
  if (rc) return rc;
  rc = upload(ws + 256 * 1024, bias, sizeof(bias), st);
  if (rc) return rc;
  Layer L;
  rc = build_deconv(L, x_bf16, B, h, w, ws, reinterpret_cast<const float*>(ws + 256 * 1024), y_bf16, block_layout ? 0 : 1);
  if (rc) return rc;
  rc = launch_layer(L, st);
  if (rc) return rc;
  return cuda_status(cudaStreamSynchronize(st));
}

// x2 geometry (SRFBN's k6 s2 p2, config C4), one layer each through the kernels the plan uses:
//   up = 1: ConvTranspose2d(32,32,6,2,2) + PReLU, x (B,h,w,32) -> y (B,2h,2w,32), w_host (32 in, 32 out, 6, 6)
//   up = 0: Conv2d(32,32,6,2,2) + PReLU, x (B,2h,2w,32) -> y (B,h,w,32), w_host (32 out, 32 in, 6, 6)
extern "C" int vsr_test_x2_layer(const void* x_bf16, int up, int B, int h, int w, const float* w_host,
                                 const float* b_host, float slope, void* y_bf16, void* workspace,
                                 size_t workspace_bytes, vsr_stream_t stream) {
  if (!x_bf16 || !w_host || !b_host || !y_bf16 || !workspace || B <= 0 || h <= 0 || w <= 0) return VSR_ERR_INVALID_ARG;
  if (workspace_bytes < vsr_test_workspace_bytes(B, h, w)) return VSR_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  std::vector<uint16_t> wp((size_t)36 * 32 * 32);
  if (up) pack_deconv2(w_host, wp.data());
  else pack_downconv2(w_host, wp.data());
  float bias[33];
  memcpy(bias, b_host, 32 * 4);
  bias[32] = slope;
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  int rc = upload(ws, wp.data(), wp.size() * 2, st);
  if (rc) return rc;
  rc = upload(ws + 256 * 1024, bias, sizeof(bias), st);
  if (rc) return rc;
  Layer L;
  const float* bdev = reinterpret_cast<const float*>(ws + 256 * 1024);
  rc = up ? build_deconv2(L, x_bf16, B, h, w, ws, bdev, y_bf16) : build_downconv2(L, x_bf16, B, h, w, ws, bdev, y_bf16);
  if (rc) return rc;
  rc = launch_layer(L, st);
  if (rc) return rc;
  return cuda_status(cudaStreamSynchronize(st));
}

// downtran (nsrc >= 2; wt (32, 32*nsrc) fp32 host, bt (32), slope_t) + PReLU + Conv2d(32,32,8,4,2) (wd (32,32,8,8),
// bd (32), slope_d) + PReLU through the fused kernel and finalize_lr_kernel.  hr: nsrc maps in block layout,
// contiguous (nsrc, B, h+1, w+1, 16, 32) BF16.  y (B,h,w,32) BF16.  workspace additionally holds the fp32
// partial-sum slots: vsr_test_workspace_bytes(B,h,w) + B*h*w*512 bytes.
extern "C" int vsr_test_fused_down(const void* hr_bf16, int nsrc, int B, int h, int w, const float* wt_host,
                                   const float* bt_host, float slope_t, const float* wd_host, const float* bd_host,
                                   float slope_d, void* y_bf16, void* workspace, size_t workspace_bytes,
                                   vsr_stream_t stream) {
  if (!hr_bf16 || !wd_host || !bd_host || !y_bf16 || !workspace || B <= 0 || h <= 0 || w <= 0 || nsrc < 1 || nsrc > 6)
    return VSR_ERR_INVALID_ARG;
  if (nsrc > 1 && (!wt_host || !bt_host)) return VSR_ERR_INVALID_ARG;
  const size_t base_bytes = vsr_test_workspace_bytes(B, h, w);
  const size_t acc_bytes = (size_t)B * h * w * 512;
  if (workspace_bytes < base_bytes + acc_bytes) return VSR_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  std::vector<uint16_t> wd((size_t)128 * 512);
  pack_downconv_fused(wd_host, wd.data());
  int rc = upload(ws, wd.data(), wd.size() * 2, st);
  if (rc) return rc;
  float bd[33], bt[33];
  memcpy(bd, bd_host, 32 * 4);
  bd[32] = slope_d;
  rc = upload(ws + 256 * 1024, bd, sizeof(bd), st);
  if (rc) return rc;
  if (nsrc > 1) {
    std::vector<uint16_t> wt((size_t)32 * 32 * nsrc);
    pack_pointwise(wt_host, 32, 32 * nsrc, wt.data());
    rc = upload(ws + 160 * 1024, wt.data(), wt.size() * 2, st);
    if (rc) return rc;
    memcpy(bt, bt_host, 32 * 4);
    bt[32] = slope_t;
    rc = upload(ws + 257 * 1024, bt, sizeof(bt), st);
    if (rc) return rc;
  }
  float* acc = reinterpret_cast<float*>(ws + base_bytes);
  const void* hrs[6];
  const size_t plane = (size_t)B * (h + 1) * (w + 1) * 16 * 64;
  for (int j = 0; j < nsrc; ++j) hrs[j] = reinterpret_cast<const uint8_t*>(hr_bf16) + j * plane;
  Layer L;
  rc = build_fused_down(L, hrs, nsrc, B, h, w, ws + 160 * 1024, reinterpret_cast<const float*>(ws + 257 * 1024), ws,
                        reinterpret_cast<const float*>(ws + 256 * 1024), acc, y_bf16);
  if (rc) return rc;
  rc = launch_layer(L, st);
  if (rc) return rc;
  rc = build_finalize(L, acc, reinterpret_cast<const float*>(ws + 256 * 1024), y_bf16, (int64_t)B * h * w, h, w);
  if (rc) return rc;
  rc = launch_layer(L, st);
  if (rc) return rc;
  return cuda_status(cudaStreamSynchronize(st));
}

// One feedback group with its transposed conv inside (fused_updown_kernel + finalize_lr_kernel, the plan's two launches
// for groups 3-5): ConvTranspose2d(32,32,8,4,2) (wu (32 in,32 out,8,8), bu, slope_u) + PReLU of lr (B,h,w,32) is source
// nsrc-1; downtran over hr[0..nsrc-1] (wt (32,32*nsrc), bt, slope_t) + PReLU + Conv2d(32,32,8,4,2) (wd, bd, slope_d) +
// PReLU -> y (B,h,w,32).  hr: nsrc slots (nsrc,B,8,h+1,w+1,64) in block layout; slots 0..nsrc-2 are read, slot nsrc-1
// receives the transposed conv's output iff store.  Packed operands in the first 512 KB of the workspace: wd [0, 128K),
// wt at 160K, biases at 256K / 257K / 258K (down, downtran, up), wu [384K, 512K); then the fp32 partial-sum slots.
extern "C" int vsr_test_fused_updown(const void* lr_bf16, void* hr_bf16, int nsrc, int store, int B, int h, int w,
                                     const float* wu_host, const float* bu_host, float slope_u, const float* wt_host,
                                     const float* bt_host, float slope_t, const float* wd_host, const float* bd_host,
                                     float slope_d, void* y_bf16, void* workspace, size_t workspace_bytes,
                                     vsr_stream_t stream) {
  if (!lr_bf16 || !hr_bf16 || !wu_host || !bu_host || !wt_host || !bt_host || !wd_host || !bd_host || !y_bf16 ||
      !workspace || B <= 0 || h <= 0 || w <= 0 || nsrc < 2 || nsrc > 6)
    return VSR_ERR_INVALID_ARG;
  const size_t base_bytes = vsr_test_workspace_bytes(B, h, w);
  const size_t acc_bytes = (size_t)B * h * w * 512;
  if (workspace_bytes < base_bytes + acc_bytes) return VSR_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  std::vector<uint16_t> wd((size_t)128 * 512), wu((size_t)512 * 128), wt((size_t)32 * 32 * nsrc);
  pack_downconv_fused(wd_host, wd.data());
  pack_deconv(wu_host, wu.data());
  pack_pointwise(wt_host, 32, 32 * nsrc, wt.data());
  float bd[33], bt[33], bu[33];
  memcpy(bd, bd_host, 32 * 4);
  bd[32] = slope_d;
  memcpy(bt, bt_host, 32 * 4);
  bt[32] = slope_t;
  memcpy(bu, bu_host, 32 * 4);
  bu[32] = slope_u;
  int rc = upload(ws, wd.data(), wd.size() * 2, st);
  if (!rc) rc = upload(ws + 160 * 1024, wt.data(), wt.size() * 2, st);
  if (!rc) rc = upload(ws + 384 * 1024, wu.data(), wu.size() * 2, st);
  if (!rc) rc = upload(ws + 256 * 1024, bd, sizeof(bd), st);
  if (!rc) rc = upload(ws + 257 * 1024, bt, sizeof(bt), st);
  if (!rc) rc = upload(ws + 258 * 1024, bu, sizeof(bu), st);
  if (rc) return rc;
  float* acc = reinterpret_cast<float*>(ws + base_bytes);
  const void* hrs[6];
  const size_t plane = (size_t)B * (h + 1) * (w + 1) * 16 * 64;
  for (int j = 0; j < nsrc; ++j) hrs[j] = reinterpret_cast<const uint8_t*>(hr_bf16) + j * plane;
  if (!store) hrs[nsrc - 1] = nullptr;   // as in the plan: the kernel must not touch the slot
  const float* bd_dev = reinterpret_cast<const float*>(ws + 256 * 1024);
  const float* bt_dev = reinterpret_cast<const float*>(ws + 257 * 1024);
  const float* bu_dev = reinterpret_cast<const float*>(ws + 258 * 1024);
  Layer L;
  rc = build_fused_updown(L, lr_bf16, hrs, nsrc, store, B, h, w, ws + 384 * 1024, bu_dev, ws + 160 * 1024, bt_dev, ws,
                          bd_dev, acc, y_bf16);
  if (rc) return rc;
  rc = launch_layer(L, st);
  if (rc) return rc;
  rc = build_finalize(L, acc, bd_dev, y_bf16, (int64_t)B * h * w, h, w);
  if (rc) return rc;
  rc = launch_layer(L, st);
  if (rc) return rc;
  return cuda_status(cudaStreamSynchronize(st));
}
