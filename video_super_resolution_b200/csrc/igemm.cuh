// igemm.cuh -- one persistent, warp-specialised implicit-GEMM kernel (tcgen05 + TMEM + TMA) that
// serves every dense layer of the fusion stack (SURVEY.md Appendix C):
//
//     D[128 pixels, BN] = sum over K-chunks  A_chunk[128, CK] * W_chunk[BN, CK]^T      (BF16 -> FP32)
//
//   * an A chunk is a TMA box [CK channels, tile_w, tile_h, 1] of a channels-last activation
//     tensor at (c0, x0+dx, y0+dy, b): 1x1 convs use one chunk per 32-channel slice of each
//     concatenated source (torch.cat disappears), the 8x8-s4 transposed conv uses the 2x2 LR
//     taps, the 8x8-s4 conv the 2x2 blocks of the "HR block" layout, the 3x3 conv its 9 taps;
//     TMA's out-of-bounds zero fill IS the zero padding of the convolutions;
//   * the weights of the layer (<=128 KB) are loaded once per CTA and stay resident in smem;
//   * warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM alloc), warps 2-5 = epilogue
//     (tcgen05.ld -> bias + PReLU -> BF16 -> global), accumulators double-buffered in TMEM so the
//     epilogue of tile i overlaps the MMAs of tile i+1.
//
// Layout conventions are documented in DESIGN.md ("HR block layout").
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"

namespace vsr {

constexpr int kTileM = 128;          // UMMA M
constexpr int kMaxChunks = 72;       // K chunks per tile (downconv: 32 with CK=64, 64 with CK=32)
constexpr int kMaxSources = 6;       // concatenated A sources (downtran of group 5)
constexpr int kMaxStages = 16;
constexpr int kIgemmThreads = 192;   // 6 warps: producer, MMA, 4 epilogue (EPI_ROWS / EPI_CONV_OUT)
constexpr int kDeconvEpiWarps = 16;  // EPI_DECONV: 4 warps per TMEM lane quarter, 2 sub-positions each
constexpr int kDeconvThreads = 64 + 32 * kDeconvEpiWarps;
constexpr int kConvOutPitch = 33;                          // floats per row of the tap-partial exchange buffer
constexpr int kConvOutStageBytes = 2 * 128 * kConvOutPitch * 4;

enum EpiMode : int;
__host__ __device__ constexpr int igemm_threads(int mode);
enum EpiMode : int {
  EPI_ROWS = 0,        // BN=32: 64-byte BF16 row per pixel at out + row*pitch + off
  EPI_DECONV = 1,      // BN=256 (one half of the 16 sub-positions): HR block layout or plain NHWC HR
  EPI_CONV_OUT = 2,    // BN=32 (27 real = 9 taps x 3): output-shift 3x3 conv, fp32 planar output + skip + mean shifts
  EPI_DECONV2 = 3,     // BN=128 (4 sub-positions x 32): x2 transposed conv k6 s2 p2, plain NHWC HR output
  EPI_DOWN2 = 4,       // BN=96 (3 column taps x 32): x2 strided conv k6 s2 p2 with the column taps in output-shift form
};

constexpr int kDown2EpiWarps = 8;    // EPI_DOWN2 / EPI_DECONV2: 2 warps per TMEM lane quarter (16 of the 32 channels / one ry each)
constexpr int kDeconv2StageBytes = kDown2EpiWarps * 32 * 128;   // EPI_DECONV2: per warp 32 LR pixels x one HR pixel pair
// threads of an igemm CTA: producer warp + MMA warp + the mode's epilogue warps
__host__ __device__ constexpr int igemm_threads(int mode) {
  return (mode == EPI_DECONV) ? kDeconvThreads : (mode == EPI_DOWN2 || mode == EPI_DECONV2) ? 64 + 32 * kDown2EpiWarps : kIgemmThreads;
}

struct Chunk {
  int8_t map;   // index into a_maps
  int8_t dx;    // spatial offset of the box origin, in pixels of the source
  int8_t dy;
  int8_t pad;
  int32_t c0;   // channel (innermost) offset
  int32_t a_off;  // byte offset of this chunk's [128 x CK] A operand inside its pipeline stage
  int32_t tx;     // bytes the chunk's TMA box brings (0: no load -- the operand is a shifted view of
                  // another chunk's box: a tap one image row down is the same box 16 rows = 16*2*CK bytes in)
};

struct alignas(64) IgemmParams {
  CUtensorMap a_maps[kMaxSources];
  CUtensorMap b_map;
  CUtensorMap out_map;         // EPI_DECONV block layout: 4-D (64 el, w+1, h+1, 8 pairs * B), box (64,16,2,1), 128B swizzle
  Chunk chunks[kMaxChunks];
  int32_t num_chunks;
  int32_t cps;                 // K chunks per pipeline stage (one barrier round trip per stage, not per chunk)
  int32_t stage_bytes;         // bytes of one pipeline stage (multiple of 1024)
  int32_t num_stages;
  // tile grid: total tiles = n_tiles * tiles_x * tiles_y * batch, n fastest
  int32_t n_tiles, tiles_x, tiles_y, batch;
  int32_t tile_w, tile_h;      // tile stride in pixels (== tile size except EPI_CONV_OUT, whose 16x8 tiles overlap)
  int32_t org_x, org_y;        // origin of tile (0,0)
  // epilogue
  const float* bias;           // [bias_n] fp32 biases, then extras: [bias_n] = PReLU slope,
                               // EPI_CONV_OUT: [bias_n+1..+3] = sub_mean bias, [bias_n+4..+6] = add_mean bias
  int32_t bias_n;
  int32_t act;                 // 1 = PReLU, 0 = identity
  void* out;
  int64_t out_pitch;           // bytes between consecutive output rows/pixels (EPI_ROWS)
  int64_t out_off;             // byte offset inside a row (channel slice of a concat buffer)
  int64_t flat_rows;           // >0: flat mode, rows are linear (tile_h == 1); else spatial
  int32_t out_h, out_w;        // spatial extent of valid output rows (spatial mode)
  int32_t lr_h, lr_w;          // LR size (block-layout masks, deconv geometry)
  int32_t hrb_mask;            // EPI_ROWS flat over the HR block layout: zero the padding ring
  int32_t deconv_nhwc;         // EPI_DECONV: 1 = write plain NHWC HR instead of the block layout
  // EPI_CONV_OUT extras
  const float* skip_src;       // network input x (M,3,h,w) fp32
  float inv_scale;             // 1 / upscale factor of the bilinear skip (0.25 or 0.5)
};

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// one arrival per warp: 512 epilogue threads arriving one by one are 512 serialised shared-memory atomics on one
// word per hand-over (~32 cycles per warp, B300_MICROARCH "ATOMS single-bank"); the warp synchronises first
// (every lane has executed its tcgen05.fence / fence.proxy.async), then one lane arrives for all
__device__ __forceinline__ void mbar_arrive_warp(uint64_t* bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(addr),
      "r"(parity)
      : "memory");
}
// the same wait with the retry loop in C++ instead of inside the asm: the fused kernel's epilogue waits were
// tuned in this form, and mbar_wait there compiles to different code (one more register, ~90 more instructions)
__device__ __forceinline__ void mbar_wait_poll(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// TMA store: shared (128B-swizzled tile) -> global, completion tracked by the thread's bulk groups
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
// tcgen05.commit: arrives on the mbarrier when all previously issued MMAs of this thread retire
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same, accumulate flag as an immediate predicate (unrolled issue loops)
template <bool kAccumulate>
__device__ __forceinline__ void umma_bf16_imm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "n"(kAccumulate ? 1 : 0)
      : "memory");
}
// one lane of a converged warp
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "elect.sync _|P, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, swizzled shared-memory matrix descriptor (PTX "matrix descriptor", sm_100 version 1):
// bits [0,14) start>>4, [16,30) LBO>>4 (unused for swizzled K-major: 1), [32,46) SBO>>4 = bytes
// between 8-row groups, [46,48) version=1, [61,64) layout (2 = 128B swizzle, 4 = 64B swizzle).
template <int kSwizzleBytes>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  constexpr uint64_t layout = (kSwizzleBytes == 128) ? 2ull : 4ull;
  constexpr uint64_t sbo = (8ull * kSwizzleBytes) >> 4;
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (sbo << 32) | (1ull << 46) | (layout << 61);
}
// kind::f16 instruction descriptor: D=F32 (bits 4-5 = 1), A=B=BF16 (bits 7-9, 10-12 = 1), both
// K-major (bits 15,16 = 0), N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ constexpr uint32_t make_idesc(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
}

// 256-bit global store (sm_100): one full 32-byte sector per lane instead of two half-written ones
__device__ __forceinline__ void stg_v8(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t e, uint32_t f,
                                       uint32_t g, uint32_t h) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d), "r"(e),
               "r"(f), "r"(g), "r"(h)
               : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float prelu(float v, float slope, int act) { return (act && v < 0.0f) ? v * slope : v; }
// Two activations at once: round to BF16, then PReLU in packed BF16.  For a slope in [0,1]
// PReLU(x) = max(x, slope*x); for a slope > 1 it is min(x, slope*x); a negative slope needs the
// general form max(x,0) + slope*min(x,0).  The slope is uniform per layer, so the form is chosen
// once per kernel (`mode`) and the common case costs 2 packed instructions per pair.
struct PreluCfg {
  __nv_bfloat162 slope2;
  int mode;   // 0: max(x, s*x)   1: min(x, s*x)   2: general   3: identity
};
__device__ __forceinline__ PreluCfg make_prelu(float slope, int act) {
  PreluCfg c;
  c.slope2 = __floats2bfloat162_rn(slope, slope);
  c.mode = !act ? 3 : (slope >= 0.0f && slope <= 1.0f) ? 0 : (slope > 1.0f ? 1 : 2);
  return c;
}
__device__ __forceinline__ uint32_t prelu_pack(float a, float b, const PreluCfg& c) {
  const __nv_bfloat162 x = __floats2bfloat162_rn(a, b);
  __nv_bfloat162 r;
  if (c.mode == 0) {
    r = __hmax2(x, __hmul2(x, c.slope2));
  } else if (c.mode == 3) {
    r = x;
  } else if (c.mode == 1) {
    r = __hmin2(x, __hmul2(x, c.slope2));
  } else {
    const __nv_bfloat162 z = __floats2bfloat162_rn(0.0f, 0.0f);
    r = __hfma2(__hmin2(x, z), c.slope2, __hmax2(x, z));
  }
  return *reinterpret_cast<const uint32_t*>(&r);
}
// 32 accumulator columns -> 16 packed BF16 pairs with bias (fp32 add) and PReLU
__device__ __forceinline__ void convert32(const uint32_t (&v)[32], const float* bias, const PreluCfg& c,
                                          uint32_t (&o)[16]) {
  const float4* b4 = reinterpret_cast<const float4*>(bias);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 bb = b4[j];
    o[2 * j] = prelu_pack(__uint_as_float(v[4 * j]) + bb.x, __uint_as_float(v[4 * j + 1]) + bb.y, c);
    o[2 * j + 1] = prelu_pack(__uint_as_float(v[4 * j + 2]) + bb.z, __uint_as_float(v[4 * j + 3]) + bb.w, c);
  }
}
// 16 accumulator columns -> 8 packed BF16 pairs
__device__ __forceinline__ void convert16(const uint32_t (&v)[16], const float* bias, const PreluCfg& c,
                                          uint32_t (&o)[8]) {
  const float4* b4 = reinterpret_cast<const float4*>(bias);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 bb = b4[j];
    o[2 * j] = prelu_pack(__uint_as_float(v[4 * j]) + bb.x, __uint_as_float(v[4 * j + 1]) + bb.y, c);
    o[2 * j + 1] = prelu_pack(__uint_as_float(v[4 * j + 2]) + bb.z, __uint_as_float(v[4 * j + 3]) + bb.w, c);
  }
}
__device__ __forceinline__ void zero16(uint32_t (&o)[16]) {
#pragma unroll
  for (int j = 0; j < 16; ++j) o[j] = 0u;
}

struct TileCoord {
  int n_tile, x0, y0, b;
};
// Tile walk of a persistent CTA: tile = blockIdx.x + k * gridDim.x, decoded as (n fastest, x, y, b).  The
// decode costs four divisions by run-time values (~150 dependent instructions); done per tile by the single
// producer thread and by every epilogue warp it was a visible part of the per-tile floor of the thin layers
// (deconv: ~1 us per tile).  The walk divides once and then advances by the constant stride with carries.
struct TileWalk {
  int n, x, y, b;            // current tile, in tile units
  int sn, sx, sy, sb;        // gridDim.x decomposed in the same radix
  __device__ __forceinline__ void init(const IgemmParams& p, int tile, int stride) {
    n = tile % p.n_tiles;
    int r = tile / p.n_tiles;
    x = r % p.tiles_x;
    r /= p.tiles_x;
    y = r % p.tiles_y;
    b = r / p.tiles_y;
    sn = stride % p.n_tiles;
    r = stride / p.n_tiles;
    sx = r % p.tiles_x;
    r /= p.tiles_x;
    sy = r % p.tiles_y;
    sb = r / p.tiles_y;
  }
  __device__ __forceinline__ void next(const IgemmParams& p) {
    n += sn;
    int c = 0;
    if (n >= p.n_tiles) { n -= p.n_tiles; c = 1; }
    x += sx + c;
    c = 0;
    if (x >= p.tiles_x) { x -= p.tiles_x; c = 1; }
    y += sy + c;
    c = 0;
    if (y >= p.tiles_y) { y -= p.tiles_y; c = 1; }
    b += sb + c;
  }
  __device__ __forceinline__ TileCoord coord(const IgemmParams& p) const {
    TileCoord t;
    t.n_tile = n;
    t.x0 = x * p.tile_w + p.org_x;
    t.y0 = y * p.tile_h + p.org_y;
    t.b = b;
    return t;
  }
};

// smem carve-up (dynamic, base aligned to 1024 by the kernel):
//   [0, num_chunks*BN*CK*2)            resident weights, one swizzled [BN, CK] block per K chunk
//   [.., + stages*128*CK*2)            A ring
//   then barriers / tmem pointer / bias
template <int CK, int BN>
__host__ __device__ constexpr int b_chunk_bytes() { return BN * CK * 2; }
template <int CK>
__host__ __device__ constexpr int a_stage_bytes() { return kTileM * CK * 2; }

constexpr int kDeconvStageBytes = kDeconvEpiWarps * 32 * 128;   // EPI_DECONV: per warp 32 blocks x 2 sub-positions x 64 B

template <int CK, int BN>
inline size_t igemm_smem_bytes(int num_chunks, size_t ring_bytes, int extra = 0) {
  size_t b = (size_t)num_chunks * b_chunk_bytes<CK, BN>();
  b = (b + 1023) / 1024 * 1024;
  return 1024 /*align slack*/ + b + ring_bytes + 1024 /*barriers + bias*/ + 2048 + extra;
}

template <int MODE, int CK, int BN>
__global__ void __launch_bounds__(igemm_threads(MODE), 1)
igemm_kernel(const __grid_constant__ IgemmParams p) {
  constexpr int kThreadsHere = igemm_threads(MODE);
  constexpr int kEpiThreads = kThreadsHere - 64;
  static_assert(CK == 32 || CK == 64, "K chunk is 32 (64B swizzle) or 64 (128B swizzle) BF16");
  static_assert(BN == 16 || BN == 32 || BN == 96 || BN == 128 || BN == 256, "supported N tiles");
  constexpr int kSwz = CK * 2;
  // accumulator stages: two; four for the x2 layers, whose MMA time per tile (~1150 cycles) is of the order of one
  // commit -> wake -> tcgen05.ld -> arrive -> wake round trip, so with two the issuer and the epilogue took turns
  // (each waited ~45 % of the time on the other).  Only for kernels that are alone on their SM (512 columns).
  constexpr int kAccStages = (MODE == EPI_DECONV2 || MODE == EPI_DOWN2) ? 4 : 2;
  constexpr int kTmemCols = (kAccStages * BN <= 32) ? 32 : (kAccStages * BN <= 64) ? 64 : (kAccStages * BN <= 128) ? 128
                          : (kAccStages * BN <= 256) ? 256 : 512;
  static_assert(kAccStages * BN <= 512, "TMEM columns");
  constexpr int kABytes = a_stage_bytes<CK>();
  constexpr int kBBytes = b_chunk_bytes<CK, BN>();

  extern __shared__ uint8_t smem_raw[];
  // align by pointer arithmetic (an integer round trip would demote every access to generic LD/ST)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int b_region = ((p.num_chunks * kBBytes) + 1023) / 1024 * 1024;
  uint8_t* smem_b = smem;
  uint8_t* smem_a = smem + b_region;
  uint8_t* tail = smem_a + p.num_stages * p.stage_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);          // [kMaxStages]
  uint64_t* empty_bar = full_bar + kMaxStages;                     // [kMaxStages]
  uint64_t* tmem_full = empty_bar + kMaxStages;                    // [2]
  uint64_t* tmem_empty = tmem_full + 4;                            // [4]
  uint64_t* b_full = tmem_empty + 4;                               // [1]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(b_full + 1);
  float* s_bias = reinterpret_cast<float*>(tail + 512);            // up to 384 floats
  uint8_t* s_stage = tail + 2048;                                  // EPI_DECONV store staging (64 KB)

  const int cta = blockIdx.x, ncta = gridDim.x;   // persistent CTAs: tiles cta, cta + ncta, ...
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.n_tiles * p.tiles_x * p.tiles_y * p.batch;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.num_stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < kAccStages; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], kEpiThreads / 32);
    }
    mbar_init(b_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<kTmemCols>(tmem_ptr);
  constexpr int kBiasExtra = (MODE == EPI_CONV_OUT) ? 7 : 1;
  for (int i = threadIdx.x; i < p.bias_n + kBiasExtra; i += kThreadsHere) s_bias[i] = p.bias[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer (the warp walks the loop, one elected lane issues) =====================
    {
      // resident weights: every K chunk of this CTA's N tile, once
      const int n_tile0 = cta % p.n_tiles;
      if (elect_one()) {
        mbar_expect_tx(b_full, (uint32_t)(p.num_chunks * kBBytes));
        for (int kc = 0; kc < p.num_chunks; ++kc)
          tma_load_2d(smem_b + kc * kBBytes, &p.b_map, b_full, kc * CK, n_tile0 * BN);
      }
      __syncwarp();
      int s = 0;
      uint32_t phase = 0;
      TileWalk walk;
      walk.init(p, cta, ncta);
      for (int tile = cta; tile < total_tiles; tile += ncta, walk.next(p)) {
        const TileCoord t = walk.coord(p);
        for (int kc0 = 0; kc0 < p.num_chunks; kc0 += p.cps) {
          const int nk = min(p.cps, p.num_chunks - kc0);
          mbar_wait(&empty_bar[s], phase ^ 1);
          if (elect_one()) {
            uint32_t tx = 0;
            for (int j = 0; j < nk; ++j) tx += (uint32_t)p.chunks[kc0 + j].tx;
            mbar_expect_tx(&full_bar[s], tx);
            for (int j = 0; j < nk; ++j) {
              const Chunk c = p.chunks[kc0 + j];
              if (c.tx)
                tma_load_4d(smem_a + s * p.stage_bytes + c.a_off, &p.a_maps[c.map], &full_bar[s], c.c0, t.x0 + c.dx,
                            t.y0 + c.dy, t.b);
            }
          }
          __syncwarp();
          if (++s == p.num_stages) { s = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1 && MODE == EPI_DOWN2) {
    // ===================== MMA issuer, static schedule =====================
    // Two stages per tile (row parity 0 / 1), three row taps per stage, four K steps per tap: the 24 MMAs of N = 96
    // take 48 cycles each, so the generic issue loop below (~10 instructions and ~125 cycles per MMA on one thread:
    // chunk table look-ups, 64-bit descriptor arithmetic, ELECT + R2UR per operand) was the floor of this layer at
    // 0.21 tensor-pipe activity.  Here the whole warp walks the loop (warp-uniform values live in uniform registers),
    // every offset is an immediate, and one elected lane issues.
    constexpr uint32_t idesc = make_idesc(BN);
    constexpr uint32_t kRowTap = 16 * 128;          // a tap one tile row down: 16 pixel pairs of 128 bytes further in
    mbar_wait(b_full, 0);
    tc_fence_after();
    int s = 0;
    uint32_t phase = 0;
    int as = 0;
    uint32_t acc_phase = 0;
    const uint64_t dA = make_smem_desc<kSwz>(smem_u32(smem_a));
    const uint64_t dB = make_smem_desc<kSwz>(smem_u32(smem_b));
    for (int tile = cta; tile < total_tiles; tile += ncta) {
      mbar_wait(&tmem_empty[as], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
#pragma unroll
      for (int py = 0; py < 2; ++py) {
        mbar_wait(&full_bar[s], phase);
        tc_fence_after();
        const uint64_t a0 = dA + (uint64_t)((uint32_t)(s * p.stage_bytes) >> 4);
        if (elect_one()) {
#pragma unroll
          for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t ad = a0 + (uint64_t)((a * kRowTap) >> 4) + 2 * k;
              const uint64_t bd = dB + (uint64_t)(((py * 3 + a) * kBBytes) >> 4) + 2 * k;
              if (py == 0 && a == 0 && k == 0) umma_bf16_imm<false>(d_tmem, ad, bd, idesc);
              else umma_bf16_imm<true>(d_tmem, ad, bd, idesc);
            }
          umma_commit(&empty_bar[s]);
          if (py == 1) umma_commit(&tmem_full[as]);
        }
        __syncwarp();
        if (++s == p.num_stages) { s = 0; phase ^= 1; }
      }
      if (++as == kAccStages) { as = 0; acc_phase ^= 1; }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (the warp walks the loop, one elected lane issues) =====================
    // With the loop inside `if (lane == 0)` every operand of a tcgen05.mma went through ELECT + R2UR and the chunk
    // table through per-thread loads: ~10 instructions / ~125 cycles per MMA on the one thread, which is the MMA time
    // itself for N <= 128.  Walked by the converged warp the loop state is warp-uniform (uniform registers, LDCU).
    {
      constexpr uint32_t idesc = make_idesc(BN);
      mbar_wait(b_full, 0);
      tc_fence_after();
      int s = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t acc_phase = 0;
      const uint64_t dA = make_smem_desc<kSwz>(smem_u32(smem_a));
      const uint64_t dB = make_smem_desc<kSwz>(smem_u32(smem_b));
      for (int tile = cta; tile < total_tiles; tile += ncta) {
        mbar_wait(&tmem_empty[as], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
        for (int kc0 = 0; kc0 < p.num_chunks; kc0 += p.cps) {
          const int nk = min(p.cps, p.num_chunks - kc0);
          mbar_wait(&full_bar[s], phase);
          tc_fence_after();
          if (elect_one()) {
            for (int j = 0; j < nk; ++j) {
              const int kc = kc0 + j;
              const uint64_t a0 = dA + (uint64_t)((s * p.stage_bytes + p.chunks[kc].a_off) >> 4);
              const uint64_t b0 = dB + (uint64_t)((kc * kBBytes) >> 4);
#pragma unroll
              for (int k = 0; k < CK / 16; ++k) umma_bf16(d_tmem, a0 + 2 * k, b0 + 2 * k, idesc, (uint32_t)((kc | k) != 0));
            }
            umma_commit(&empty_bar[s]);                      // frees the stage when these MMAs retire
            if (kc0 + nk >= p.num_chunks) umma_commit(&tmem_full[as]);
          }
          __syncwarp();
          if (++s == p.num_stages) { s = 0; phase ^= 1; }
        }
        if (++as == kAccStages) { as = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp < 2 + kEpiThreads / 32) {
    // ===================== epilogue (warps 2..5; 2..17 for EPI_DECONV) =====================
    const int q = warp & 3;                 // TMEM lane quarter this warp may read
    const int row = q * 32 + lane;          // row of the 128-pixel tile
    int as = 0;
    uint32_t acc_phase = 0;
    TileWalk walk;
    walk.init(p, cta, ncta);
    for (int tile = cta; tile < total_tiles; tile += ncta, walk.next(p)) {
      const TileCoord t = walk.coord(p);
      mbar_wait(&tmem_full[as], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN);

      if constexpr (MODE == EPI_ROWS) {
        bool valid, zero = false;
        uint8_t* dst;
        if (p.flat_rows > 0) {
          const int64_t R = (int64_t)t.x0 + row;
          valid = R < p.flat_rows;
          dst = reinterpret_cast<uint8_t*>(p.out) + R * p.out_pitch + p.out_off;
          if (p.hrb_mask) {
            const int s16 = (int)(R & 15);
            const int64_t blk = R >> 4;
            const int X = (int)(blk % (p.lr_w + 1));
            const int Y = (int)((blk / (p.lr_w + 1)) % (p.lr_h + 1));
            const int ry = s16 >> 2, rx = s16 & 3;
            zero = (Y == 0 && ry < 2) || (Y == p.lr_h && ry >= 2) || (X == 0 && rx < 2) || (X == p.lr_w && rx >= 2);
          }
        } else {
          const int y = t.y0 + (row >> 4), x = t.x0 + (row & 15);   // spatial EPI_ROWS tiles are 16 x 8
          valid = (y < p.out_h) && (x < p.out_w);
          dst = reinterpret_cast<uint8_t*>(p.out) + (((int64_t)t.b * p.out_h + y) * p.out_w + x) * p.out_pitch + p.out_off;
        }
        const PreluCfg pc = make_prelu(s_bias[p.bias_n], p.act);
#pragma unroll 1
        for (int cg = 0; cg < BN / 32; ++cg) {
          uint32_t v[32];
          tmem_ld32(taddr + cg * 32, v);
          tmem_ld_wait();
          if (cg == BN / 32 - 1) {
            tc_fence_before();
            mbar_arrive_warp(&tmem_empty[as]);     // accumulator stage is free again
          }
          if (valid) {
            uint32_t o[16];
            if (zero) zero16(o);
            else convert32(v, s_bias + cg * 32, pc, o);
            // 256-bit stores for the wide rows (conv_in: 0.27 -> 0.20 ms per C2 pass); for the 64-byte rows of the 1x1
            // layers they measured 15 % SLOWER than four 128-bit stores (3.2 -> 3.8 ms per C2 pass)
            if constexpr (BN >= 128) {
              uint8_t* d8 = dst + cg * 64;
              stg_v8(d8, o[0], o[1], o[2], o[3], o[4], o[5], o[6], o[7]);
              stg_v8(d8 + 32, o[8], o[9], o[10], o[11], o[12], o[13], o[14], o[15]);
            } else {
              uint4* d4 = reinterpret_cast<uint4*>(dst + cg * 64);
#pragma unroll
              for (int j = 0; j < 4; ++j) d4[j] = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
            }
          }
        }
      } else if constexpr (MODE == EPI_DECONV) {
        // row = patch position (Y, X) in [0,h] x [0,w]; this N tile holds sub-positions
        // s = n_tile*8 .. n_tile*8+7 (ry = s>>2, rx = s&3), 32 output channels each.
        const int Y = t.y0 + (row >> 4), X = t.x0 + (row & 15);     // deconv tiles are 16 x 8 blocks
        const bool valid = (Y <= p.lr_h) && (X <= p.lr_w);
        const int H = 4 * p.lr_h, W = 4 * p.lr_w;
        const PreluCfg pc = make_prelu(s_bias[p.bias_n], 1);
        const int sub = (warp - 2) >> 2;             // which pair of sub-positions this warp converts
        if (p.deconv_nhwc) {
#pragma unroll 1
          for (int c2 = 0; c2 < 2; ++c2) {
            const int cg = sub * 2 + c2;
            uint32_t v[32];
            tmem_ld32(taddr + cg * 32, v);
            tmem_ld_wait();
            if (c2 == 1) {
              tc_fence_before();
              mbar_arrive_warp(&tmem_empty[as]);
            }
            const int s16 = t.n_tile * 8 + cg;
            const int ry = s16 >> 2, rx = s16 & 3;
            const int Yt = 4 * Y + ry - 2, Xt = 4 * X + rx - 2;       // true HR coordinates
            if (valid && (Yt >= 0) && (Yt < H) && (Xt >= 0) && (Xt < W)) {
              uint32_t o[16];
              convert32(v, s_bias, pc, o);
              uint4* d4 = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(p.out) + (((int64_t)t.b * H + Yt) * W + Xt) * 64);
#pragma unroll
              for (int j = 0; j < 4; ++j) d4[j] = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
            }
          }
        } else {
          // Block layout: this warp owns 128 contiguous bytes (2 sub-positions x 32 ch) of each of its
          // 32 block rows.  It stages them in shared memory as a [32 rows x 128 B] tile in the canonical
          // 128B-swizzle pattern and hands the tile to the TMA engine: one bulk tensor store writes two
          // contiguous 2 KB runs of the pair's plane, clips at the tensor edge, and costs the LSU
          // nothing (the first version read the tile back with LDS and stored with STG: L1TEX 70 % busy).
          uint8_t* stg = s_stage + (warp - 2) * (32 * 128);
#pragma unroll
          for (int c2 = 0; c2 < 2; ++c2) {
            const int cg = sub * 2 + c2;
            uint32_t v[32];
            tmem_ld32(taddr + cg * 32, v);
            tmem_ld_wait();
            if (c2 == 1) {
              tc_fence_before();
              mbar_arrive_warp(&tmem_empty[as]);
            }
            const int s16 = t.n_tile * 8 + cg;
            const int ry = s16 >> 2, rx = s16 & 3;
            const int Yt = 4 * Y + ry - 2, Xt = 4 * X + rx - 2;
            const bool inside = (Yt >= 0) && (Yt < H) && (Xt >= 0) && (Xt < W);   // else: zero ring
            uint32_t o[16];
            convert32(v, s_bias, pc, o);
            if (__builtin_expect(!inside, 0)) zero16(o);   // ring positions (tile border only) stay zero
            if (c2 == 0) {   // the previous tile's store must have read the staging tile before it is overwritten
              if (elect_one()) tma_store_wait_read();   // (waited for here, after the TMEM read + conversion, not before)
              __syncwarp();
            }
            uint8_t* srow = stg + lane * 128;
            const int sw = lane & 7;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              *reinterpret_cast<uint4*>(srow + (((c2 * 4 + j) ^ sw) << 4)) =
                  make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
          }
          fence_async_smem();
          __syncwarp();
          if (elect_one()) {   // (the same lane every time: bulk groups are per thread)
            // one box = this warp's 2 block rows x 16 blocks of one sub-position-pair plane; rows or
            // columns beyond the tensor edge are clipped by the TMA unit
            if (t.y0 + 2 * q <= p.lr_h)
              tma_store_4d(&p.out_map, stg, 0, t.x0, t.y0 + 2 * q, t.b * 8 + t.n_tile * 4 + sub);
            tma_store_commit();
          }
        }
      } else if constexpr (MODE == EPI_DECONV2) {
        // ConvTranspose2d k6 s2 p2 (SRFBN's x2 geometry): row = LR pixel (Y,X), the 3x3 LR taps are the
        // K chunks, column group s = ry*2+rx is HR pixel (2Y+ry, 2X+rx).  8 epilogue warps, 2 per TMEM lane quarter:
        // a warp converts both rx of one ry, i.e. the 128 contiguous bytes (HR pixel pair) of each of its 32 LR
        // pixels, stages them as a [32 x 128 B] tile in the 128B-swizzle pattern and stores each of its two tile rows
        // with one TMA bulk tensor store (16 pairs = 2 KB contiguous; clipped at the tensor edge).  The version that
        // stored from registers (a 16-byte piece per lane at a 128-byte stride: 32 partial sectors per instruction)
        // spent half of the layer's time in the LSU: 70.6 ms per C4 pass, 36 ms with the stores knocked out.
        const PreluCfg pc = make_prelu(s_bias[p.bias_n], 1);
        const int ry = (warp - 2) >> 2;
        uint8_t* stg = s_stage + (warp - 2) * (32 * 128);
#pragma unroll
        for (int rx = 0; rx < 2; ++rx) {
          uint32_t v[32];
          tmem_ld32(taddr + (ry * 2 + rx) * 32, v);
          tmem_ld_wait();
          if (rx == 1) {
            tc_fence_before();
            mbar_arrive_warp(&tmem_empty[as]);
          }
          uint32_t o[16];
          convert32(v, s_bias, pc, o);
          if (rx == 0) {   // the previous tile's stores must have read the staging tile before it is overwritten
            if (elect_one()) tma_store_wait_read();
            __syncwarp();
          }
          uint8_t* srow = stg + lane * 128;
          const int sw = lane & 7;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            *reinterpret_cast<uint4*>(srow + (((rx * 4 + j) ^ sw) << 4)) =
                make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
        }
        fence_async_smem();
        __syncwarp();
        if (elect_one()) {
          const int Yq = t.y0 + 2 * q;
          tma_store_4d(&p.out_map, stg, 0, t.x0, 2 * Yq + ry, t.b);
          tma_store_4d(&p.out_map, stg + 16 * 128, 0, t.x0, 2 * (Yq + 1) + ry, t.b);
          tma_store_commit();
        }
      } else if constexpr (MODE == EPI_DOWN2) {
        // Conv2d k6 s2 p2 (SRFBN's x2 geometry) with the three column taps b = kx>>1 in output-shift form: row =
        // pixel-pair column x' = x0 + xi of LR row Y, accumulator columns [b*32, b*32+32) hold
        // P_b[Y, x'] = sum over (ky, px, c) of HR[2(Y + (ky>>1) - 1) + (ky&1), 2x' + px, c] * W[o, c, ky, 2b + px], and
        // out[Y, X] = P_0[Y, X-1] + P_1[Y, X] + P_2[Y, X+1]: every HR pixel is loaded once per tile (1.25 x 16/14 with
        // the row halo and the overlapping columns) instead of once per column tap.  A TMEM lane quarter is two tile
        // rows of 16 columns, so the neighbours are the adjacent lanes; columns 1..14 of a tile are finished.
        const int xi = row & 15;
        const int Y = t.y0 + (row >> 4), X = t.x0 + xi;
        const bool valid = (xi >= 1) && (xi <= 14) && (Y < p.out_h) && (X < p.out_w);
        const PreluCfg pc = make_prelu(s_bias[p.bias_n], p.act);
        // 8 epilogue warps, 2 per TMEM lane quarter: each finishes 16 of the 32 channels (with 4 warps doing all 32
        // the epilogue was busy 79 % of the time and the MMA issuer waited for accumulators)
        const int half = (warp - 2) >> 2;
        uint32_t acc[16], vl[16], vr[16];
        tmem_ld16(taddr + 32 + 16 * half, acc);
        tmem_ld16(taddr + 16 * half, vl);
        tmem_ld16(taddr + 64 + 16 * half, vr);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive_warp(&tmem_empty[as]);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float l = __shfl_up_sync(0xffffffffu, __uint_as_float(vl[j]), 1);
          const float r = __shfl_down_sync(0xffffffffu, __uint_as_float(vr[j]), 1);
          acc[j] = __float_as_uint((__uint_as_float(acc[j]) + l) + r);
        }
        if (valid) {
          uint32_t o[8];
          convert16(acc, s_bias + 16 * half, pc, o);
          uint4* d4 = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(p.out) +
                                               (((int64_t)t.b * p.out_h + Y) * p.out_w + X) * p.out_pitch + p.out_off +
                                               32 * half);
          d4[0] = make_uint4(o[0], o[1], o[2], o[3]);      // (one 256-bit store instead: same-box A/B neutral)
          d4[1] = make_uint4(o[4], o[5], o[6], o[7]);
        }
      } else {  // EPI_CONV_OUT
        // 3x3 conv in "output-shift" form: row = INPUT pixel (xi, yi) of a 16x8 tile whose origin is
        // (x0, y0) = 14*tx-1, 6*ty-1; D[row, (ky*3+kx)*3 + o] = sum_c in[row, c] * W[o, c, ky, kx] is the
        // contribution of this pixel to output (y - ky + 1, x - kx + 1).  Every input pixel is loaded
        // once per tile (1.5x overlap) instead of once per tap (9x); the 27 partials are exchanged
        // through shared memory and the 14x6 interior pixels gather their 9 neighbours.
        float* S = reinterpret_cast<float*>(s_stage) + (as * 128) * kConvOutPitch;
        {
          uint32_t v[32];
          tmem_ld32(taddr, v);
          tmem_ld_wait();
          tc_fence_before();
          mbar_arrive_warp(&tmem_empty[as]);
          float* srow = S + row * kConvOutPitch;
#pragma unroll
          for (int j = 0; j < 27; ++j) srow[j] = __uint_as_float(v[j]);
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");     // the 4 epilogue warps only
        const int xi = row & 15, yi = row >> 4;
        const int X = t.x0 + xi, Y = t.y0 + yi;
        if (xi >= 1 && xi <= 14 && yi >= 1 && yi <= 6 && X < p.out_w && Y < p.out_h) {
          float acc[3] = {s_bias[0], s_bias[1], s_bias[2]};
#pragma unroll
          for (int ky = 0; ky < 3; ++ky)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
              const float* q = S + ((yi + ky - 1) * 16 + (xi + kx - 1)) * kConvOutPitch + (ky * 3 + kx) * 3;
              acc[0] += q[0];
              acc[1] += q[1];
              acc[2] += q[2];
            }
          // bilinear xs skip, align_corners=False (SRProjectionModule.py:136; ATen
          // upsample_bilinear2d: src = (dst+0.5)/s - 0.5 clamped at 0), on sub_mean(x)
          const int h = p.lr_h, w = p.lr_w;
          float sy = fmaxf((Y + 0.5f) * p.inv_scale - 0.5f, 0.0f), sx = fmaxf((X + 0.5f) * p.inv_scale - 0.5f, 0.0f);
          int y0i = (int)sy, x0i = (int)sx;
          int y1i = y0i + (y0i < h - 1 ? 1 : 0), x1i = x0i + (x0i < w - 1 ? 1 : 0);
          float ly = sy - y0i, lx = sx - x0i, hy = 1.0f - ly, hx = 1.0f - lx;
          float* out = reinterpret_cast<float*>(p.out);
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const float* src = p.skip_src + ((int64_t)t.b * 3 + c) * h * w;
            const float sb = s_bias[p.bias_n + 1 + c];
            float v00 = __ldg(src + y0i * w + x0i) + sb, v01 = __ldg(src + y0i * w + x1i) + sb;
            float v10 = __ldg(src + y1i * w + x0i) + sb, v11 = __ldg(src + y1i * w + x1i) + sb;
            float skip = hy * (hx * v00 + lx * v01) + ly * (hx * v10 + lx * v11);
            out[(((int64_t)t.b * 3 + c) * p.out_h + Y) * p.out_w + X] = skip + acc[c] + s_bias[p.bias_n + 4 + c];
          }
        }
      }
      if (++as == kAccStages) { as = 0; acc_phase ^= 1; }
    }
    __syncwarp();
    if (MODE == EPI_DECONV2 && elect_one()) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    if (MODE == EPI_DECONV && elect_one()) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // the last tile's store
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<kTmemCols>(tmem_base);
  }
}

}  // namespace vsr
