// fused_down.cuh -- one kernel for the HR half of a feedback group:
//
//     lr[i+1] = PReLU( Conv8x8s4( PReLU( Conv1x1( cat(hr[0..i]) ) ) ) )
//     ref: FeedbackBlock.forward, SRProjectionModule.py:70-80 (downtranBlocks[i-1] then downBlocks[i]),
//          intended dense-concat dataflow (SURVEY.md Appendix C)
//
// Layer by layer this is the most expensive part of the stack in HBM bytes: the 1x1 "downtran" reads
// (i+1) HR feature maps and writes one, the 8x8-s4 conv reads it back.  Here the intermediate HR map
// never leaves the SM:
//
//   tile   = 16 x 8 blocks of the HR block layout (128 blocks = 128 UMMA rows) of one map
//   phase A (per group g of 4 sub-positions): D_A[128, 4x32] = sum_j hr_j[tile, s, :] * Wt_j^T
//            A operands: TMA boxes [32 ch, 1 s, 16, 8] of the 5-D view (c, s, Xb, Yb, map); N = 32
//   convert: epilogue warps read D_A from TMEM, add bias, PReLU, zero the padding ring, round to
//            BF16 and write the [128, 128] tile into shared memory in the 128B-swizzled K-major
//            layout the tensor core reads (fence.proxy.async), i.e. they PRODUCE phase B's A operand
//   phase B: D_B[128, 4 taps x 32] += H_g[128, 128] * Wd_g[128, 128]^T        (K = 512 over 4 groups)
//            "output-shift" form of the strided conv: block (Yb,Xb) contributes its tap-(dy,dx)
//            partial product to LR pixel (Yb-dy, Xb-dx); every block is read exactly once
//   epilogue: the four 32-channel tap partials of each block are combined across lanes (dx: shuffle by 1,
//            dy: shuffle by 16 / a 6 KB shared-memory exchange between lane quarters); 82 % of the LR
//            pixels are complete inside the tile and leave as finished BF16 (bias + PReLU); the pixels
//            of tile row 7 and of the tile's last column go to per-pixel FP32 "slots" with exactly one
//            writer each and finalize_lr_kernel sums them -- no atomics, deterministic.
//            (A first version used red.global.add.v4.f32: ~10k cycles per tile of L2 atomic
//            throughput, the kernel's fixed cost; the second sent every pixel through the slots.)
//
// HAS_TRAN = false is group 0 (no downtran: H = hr[0]); phase B's A operand then comes straight from
// TMA.  Warp roles: warp 0 TMA producer, warp 1 MMA issuer (phase A with HAS_TRAN), warps 2-17 epilogue,
// warp 18 conv-weight streamer, warp 19 phase-B MMA issuer (HAS_TRAN).
#pragma once
#include "igemm.cuh"

namespace vsr {

constexpr int kFusedEpiWarps = 16;   // 4 per TMEM lane quarter: one sub-position / one tap each
constexpr int kFusedWdWarp = 2 + kFusedEpiWarps;             // last warp: streams the conv weights
constexpr int kFusedBWarp = kFusedWdWarp + 1;                // issues the phase-B MMAs (HAS_TRAN)
constexpr int kFusedThreads = 32 * (kFusedBWarp + 1);
constexpr int kFusedMaxStages = 16;
constexpr int kWdGroupBytes = 128 * 128 * 2; // 8x8-s4 weights of one sub-position group: 2 chunks [128 n][64 k]
constexpr int kWdRingBytes = 2 * kWdGroupBytes;  // streamed per group from L2 through a 2-deep ring
constexpr int kWtChunkBytes = 32 * 32 * 2;   // one 32x32 downtran slice (64-byte rows, 64B swizzle)
constexpr int kHBytes = 128 * 128 * 2;       // phase-B A operand of one sub-position group
constexpr int kXchgBytes = 3 * 4 * 16 * 8 * 4;   // row partials handed from lane quarter q+1 to q: [3][4 subs][16 px][8 ch] fp32
constexpr int kLRBox = 16 * 9 * 64;         // fused_updown_kernel: one LR box [32 ch, 16, 9 rows] (64B swizzle)
constexpr int kLRBytes = 2 * kLRBox;         // the dx = -1 and dx = 0 boxes of a tile
constexpr int kWuTapBytes = 128 * 32 * 2;    // transposed-conv weights of one LR tap for 4 sub-positions: [128 n][32 k]

struct alignas(64) FusedDownParams {
  CUtensorMap hr_maps[kMaxSources];   // HAS_TRAN: 4-D (64, w+1, h+1, 8*B) pair planes, box (64,16,8,1) = 2 sub-positions, 128B swizzle
  CUtensorMap h0_map;                 // !HAS_TRAN: the same view of hr[0]
  CUtensorMap wt_map;                 // 2-D (32*nsrc, 32), box (32,32), 64B swizzle
  CUtensorMap wd_map;                 // 2-D (512, 128), box (64,128), 128B swizzle
  int32_t nsrc;
  int32_t num_stages;
  int32_t tiles_x, tiles_y, batch;
  int32_t lr_h, lr_w;
  const float* tran_bias;             // [32] biases + [1] PReLU slope of the downtran
  const float* down_bias;             // [32] biases + [1] PReLU slope of the strided conv
  float* part;                        // (B, h, w, 4 slots, 32) fp32 partial sums of the BOUNDARY pixels (see final epilogue)
  void* lr_out;                       // (B, h, w, 32) bf16: finished interior pixels
  // fused_updown_kernel only (hr_maps[nsrc-1] is then the store view of hr[nsrc-1])
  CUtensorMap up_map;                 // the transposed conv's input (B, h, w, 32), box (32,16,9,1), 64B swizzle
  CUtensorMap wu_map;                 // its weights 2-D (128, 512), box (32,128), 64B swizzle
  const float* up_bias;               // [32] biases + [1] PReLU slope of the transposed conv
  int32_t hr_store;                   // 1: store U into hr[nsrc-1] (a later group reads it)
};

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}

template <bool HAS_TRAN>
inline size_t fused_down_smem_bytes(int nsrc, int num_stages) {
  size_t wt = HAS_TRAN ? ((size_t)nsrc * kWtChunkBytes + 1023) / 1024 * 1024 : 0;
  size_t stage = HAS_TRAN ? 16384 : 2 * 16384;
  return 1024 + kWdRingBytes + wt + (HAS_TRAN ? kHBytes : 0) + (size_t)num_stages * stage + 1024 + kXchgBytes;
}

inline size_t fused_updown_smem_bytes(int nsrc, int num_stages) {
  return fused_down_smem_bytes<true>(nsrc, num_stages) + kLRBytes;
}

// MERGED (HAS_TRAN only): the kernel also computes the newest source hr[nsrc-1] itself (see fused_updown_kernel)
template <bool HAS_TRAN, bool MERGED>
__device__ __forceinline__ void fused_down_body(const FusedDownParams& p) {
  static_assert(HAS_TRAN || !MERGED, "the merged kernel needs phase A");
  constexpr int kStageBytes = HAS_TRAN ? 16384 : 2 * 16384;
  constexpr int kTmemCols = HAS_TRAN ? 512 : 256;
  // TMEM columns: D_A [0, 256) (two buffers, HAS_TRAN), D_B [kDB, kDB + 128 * kDBufs); MERGED: T_U [kTU, kTU + 128)
  constexpr uint32_t kDB = MERGED ? 384 : HAS_TRAN ? 256 : 0;
  constexpr int kDBToggle = MERGED ? 0 : 1;          // MERGED: one D_B buffer (tb stays 0)
  constexpr uint32_t kTU = 256;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_wd = smem;
  uint8_t* s_wt = s_wd + kWdRingBytes;
  const int wt_region = HAS_TRAN ? ((p.nsrc * kWtChunkBytes + 1023) / 1024 * 1024) : 0;
  uint8_t* s_h = s_wt + wt_region;
  uint8_t* s_lr = s_h + (HAS_TRAN ? kHBytes : 0);                // MERGED: the tile's two LR boxes
  uint8_t* s_a = s_lr + (MERGED ? kLRBytes : 0);
  uint8_t* tail = s_a + p.num_stages * kStageBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);      // [kFusedMaxStages]
  uint64_t* empty_bar = full_bar + kFusedMaxStages;            // [kFusedMaxStages]
  uint64_t* w_full = empty_bar + kFusedMaxStages;              // [1] downtran weights resident
  uint64_t* wd_full = w_full + 1;                              // [2] conv-weight ring
  uint64_t* wd_empty = wd_full + 2;                            // [2]
  uint64_t* da_full = wd_empty + 2;                            // [2]
  uint64_t* da_empty = da_full + 2;                            // [2]
  uint64_t* h_full = da_empty + 2;                             // [1]
  uint64_t* h_empty = h_full + 1;                              // [1]
  uint64_t* db_full = h_empty + 1;                             // [2]
  uint64_t* db_empty = db_full + 2;                            // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(db_empty + 2);
  uint64_t* tu_full = db_empty + 3;                            // MERGED: [1] T_U accumulated
  uint64_t* tu_empty = tu_full + 1;                            // [1] T_U read by the epilogue
  uint64_t* u_full = tu_empty + 1;                             // [1] U_g written into s_h
  uint64_t* lr_full = u_full + 1;                              // [1] LR boxes of the tile loaded
  uint64_t* lr_empty = lr_full + 1;                            // [1] LR boxes consumed (last T_U MMA of the tile)
  float* s_bias = reinterpret_cast<float*>(tail + 512);        // 33 floats: downtran bias + slope
  float* s_down = s_bias + 36;                                 // 33 floats: strided-conv bias + slope
  float* s_ubias = s_down + 36;                                // MERGED: 33 floats: transposed-conv bias + slope
  float4* s_x = reinterpret_cast<float4*>(tail + 1024);        // kXchgBytes: final-epilogue row exchange

  const int cta = blockIdx.x, ncta = gridDim.x;   // persistent CTAs: tiles cta, cta + ncta, ...
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.tiles_x * p.tiles_y * p.batch;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.num_stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(w_full, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&wd_full[s], 1);
      mbar_init(&wd_empty[s], 1);
      mbar_init(&da_full[s], 1);
      mbar_init(&da_empty[s], kFusedEpiWarps);
      mbar_init(&db_full[s], 1);
      mbar_init(&db_empty[s], kFusedEpiWarps);
    }
    mbar_init(h_full, kFusedEpiWarps);
    mbar_init(h_empty, 1);
    if (MERGED) {
      mbar_init(tu_full, 1);
      mbar_init(tu_empty, kFusedEpiWarps);
      mbar_init(u_full, 1);
      mbar_init(lr_full, 1);
      mbar_init(lr_empty, 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<kTmemCols>(tmem_ptr);
  if (HAS_TRAN)
    for (int i = threadIdx.x; i < 33; i += kFusedThreads) s_bias[i] = p.tran_bias[i];
  if (MERGED)
    for (int i = threadIdx.x; i < 33; i += kFusedThreads) s_ubias[i] = p.up_bias[i];
  for (int i = threadIdx.x; i < 33; i += kFusedThreads) s_down[i] = p.down_bias[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  auto tile_coord = [&](int tile, int& x0, int& y0, int& b) {
    x0 = (tile % p.tiles_x) * 16;
    int r = tile / p.tiles_x;
    y0 = (r % p.tiles_y) * 8;
    b = r / p.tiles_y;
  };

  if (warp == 0) {
    // ===================== TMA producer =====================
    // walked by the converged warp, one elected lane issues (as the MMA roles: the loop state stays in uniform
    // registers; "box count, not bytes, limits a single-thread producer")
    {
      if (HAS_TRAN && elect_one()) {
        mbar_expect_tx(w_full, (uint32_t)(p.nsrc * kWtChunkBytes));
        for (int j = 0; j < p.nsrc; ++j) tma_load_2d(s_wt + j * kWtChunkBytes, &p.wt_map, w_full, j * 32, 0);
      }
      __syncwarp();
      int s = 0;
      uint32_t phase = 0;
      for (int tile = cta; tile < total_tiles; tile += ncta) {
        int x0, y0, b;
        tile_coord(tile, x0, y0, b);
        for (int half = 0; half < 2; ++half) {
          if (HAS_TRAN) {
            // one box = 2 sub-positions x 128 blocks x 32 ch (16 KB): a [128 x 64] K-major tile whose K
            // halves are the two sub-positions (box count, not bytes, limits a single-thread producer)
            for (int sp = half * 8; sp < half * 8 + 8; sp += 2) {
              for (int j = 0; j < p.nsrc - (MERGED ? 1 : 0); ++j) {   // MERGED: the newest source is made on chip
                mbar_wait(&empty_bar[s], phase ^ 1);
                if (elect_one()) {
                  mbar_expect_tx(&full_bar[s], kStageBytes);
                  tma_load_4d(s_a + s * kStageBytes, &p.hr_maps[j], &full_bar[s], 0, x0, y0, b * 8 + (sp >> 1));
                }
                __syncwarp();
                if (++s == p.num_stages) { s = 0; phase ^= 1; }
              }
            }
          } else {
            for (int g = half * 2; g < half * 2 + 2; ++g) {
              mbar_wait(&empty_bar[s], phase ^ 1);
              if (elect_one()) {
                mbar_expect_tx(&full_bar[s], kStageBytes);
                tma_load_4d(s_a + s * kStageBytes, &p.h0_map, &full_bar[s], 0, x0, y0, b * 8 + 2 * g);
                tma_load_4d(s_a + s * kStageBytes + 16384, &p.h0_map, &full_bar[s], 0, x0, y0, b * 8 + 2 * g + 1);
              }
              __syncwarp();
              if (++s == p.num_stages) { s = 0; phase ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1 || (HAS_TRAN && warp == kFusedBWarp)) {
    // ===================== MMA issuers =====================
    // Timing experiments showed this role's instruction stream to be co-critical with HBM (each box costs it a
    // barrier wait, four MMA issues and a commit), so descriptors are pre-built and only offsets are added -- and the
    // loop is walked by the converged warp (its state lives in uniform registers, no ELECT + R2UR per operand as
    // inside `if (lane == 0)`), one elected lane issues.
    {
    constexpr uint32_t idesc_a = make_idesc(32);
    constexpr uint32_t idesc_b = make_idesc(128);
    if (HAS_TRAN && warp == 1) mbar_wait(w_full, 0);
    tc_fence_after();
    int s = 0;
    uint32_t phase = 0;
    uint32_t n_a[2] = {0, 0}, n_b[2] = {0, 0}, n_h = 0, n_wd = 0;
    int tb = 0;
    // matrix descriptors: the start-address field is bits [0,14) in 16-byte units, so an offset of
    // `off` bytes inside the same buffer is a plain add of off >> 4
    const uint64_t dA = make_smem_desc<128>(smem_u32(s_a));
    const uint64_t dWt = make_smem_desc<64>(smem_u32(s_wt));
    const uint64_t dH = make_smem_desc<128>(smem_u32(s_h));
    const uint64_t dWd = make_smem_desc<128>(smem_u32(s_wd));
    uint32_t n_tu = 0, n_lr = 0, n_u = 0;

    // MERGED, transposed conv of group g: T_U[128 blocks, 4 sub-positions x 32] = LR taps * Wu_g^T, K = 4 taps x 32
    // channels in igemm_kernel<EPI_DECONV>'s order (tap, then 16-wide K steps): every accumulator column gets the
    // same additions in the same order as there, N = 128 instead of 256 changes no column's sum
    auto issue_u = [&](int g) {
      constexpr uint32_t idesc_u = make_idesc(128);
      const uint64_t dLR = make_smem_desc<64>(smem_u32(s_lr));
      const uint64_t dWu = make_smem_desc<64>(smem_u32(s_wd));
      if (g == 0) mbar_wait(lr_full, n_lr & 1);
      mbar_wait(tu_empty, (n_tu & 1) ^ 1);
      mbar_wait(&wd_full[0], n_tu & 1);
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int t = 0; t < 4; ++t)
#pragma unroll
          for (int k = 0; k < 2; ++k)
            umma_bf16(tmem_base + kTU, dLR + (uint64_t)(((t & 1) * kLRBox + (t >> 1) * 1024) >> 4) + 2 * k,
                      dWu + (uint64_t)((t * kWuTapBytes) >> 4) + 2 * k, idesc_u, (uint32_t)((t | k) != 0));
        umma_commit(&wd_empty[0]);
        umma_commit(tu_full);
        if (g == 3) umma_commit(lr_empty);
      }
      __syncwarp();
      ++n_tu;
      if (g == 3) ++n_lr;
    };

    // phase A of sub-position group g: D_A[g&1] = sum_j A(s, j) * Wt_j^T for the 4 sub-positions
    auto issue_a = [&](int g) {
      const int buf = g & 1;
      mbar_wait(&da_empty[buf], (n_a[buf] & 1) ^ 1);
      tc_fence_after();
      for (int pair = 0; pair < 2; ++pair)
        for (int j = 0; j < p.nsrc - (MERGED ? 1 : 0); ++j) {
          mbar_wait(&full_bar[s], phase);
          tc_fence_after();
          const uint64_t a0 = dA + (uint64_t)((s * kStageBytes) >> 4);
          const uint64_t b0 = dWt + (uint64_t)((j * kWtChunkBytes) >> 4);
          const uint32_t d0 = tmem_base + (uint32_t)(buf * 128 + pair * 64);
          if (elect_one()) {
            const uint32_t acc = (uint32_t)(j != 0);
            umma_bf16(d0, a0, b0, idesc_a, acc);
            umma_bf16(d0, a0 + 2, b0 + 2, idesc_a, 1u);
            umma_bf16(d0 + 32, a0 + 4, b0, idesc_a, acc);
            umma_bf16(d0 + 32, a0 + 6, b0 + 2, idesc_a, 1u);
            umma_commit(&empty_bar[s]);
            if (!MERGED && pair == 1 && j == p.nsrc - 1) umma_commit(&da_full[buf]);
          }
          __syncwarp();
          if (++s == p.num_stages) { s = 0; phase ^= 1; }
        }
      if (MERGED) {
        // the last source, j = nsrc - 1, is U_g in s_h (the epilogue's conversion of T_U): the same operand bytes a TMA
        // box of hr[nsrc-1] would bring, added last into each column as before
        mbar_wait(u_full, n_u & 1);
        tc_fence_after();
        const uint64_t b0 = dWt + (uint64_t)(((p.nsrc - 1) * kWtChunkBytes) >> 4);
        if (elect_one()) {
          for (int pair = 0; pair < 2; ++pair) {
            const uint64_t a0 = dH + (uint64_t)((pair * 16384) >> 4);
            const uint32_t d0 = tmem_base + (uint32_t)(buf * 128 + pair * 64);
            umma_bf16(d0, a0, b0, idesc_a, 1u);
            umma_bf16(d0, a0 + 2, b0 + 2, idesc_a, 1u);
            umma_bf16(d0 + 32, a0 + 4, b0, idesc_a, 1u);
            umma_bf16(d0 + 32, a0 + 6, b0 + 2, idesc_a, 1u);
          }
          umma_commit(&da_full[buf]);
        }
        __syncwarp();
        ++n_u;
      }
      ++n_a[buf];
    };
    // phase B of group g: D_B[tb] += H_g * Wd_g^T
    auto issue_b = [&](int g) {
      uint64_t a0;
      if (HAS_TRAN) {
        mbar_wait(h_full, n_h & 1);
        a0 = dH;
      } else {
        mbar_wait(&full_bar[s], phase);
        a0 = dA + (uint64_t)((s * kStageBytes) >> 4);
      }
      if (g == 0) mbar_wait(&db_empty[tb], (n_b[tb] & 1) ^ 1);
      // MERGED: slot 0 of the weight ring holds the transposed-conv weights, slot 1 the conv weights
      const int wslot = MERGED ? 1 : (int)(n_wd & 1);
      mbar_wait(&wd_full[wslot], MERGED ? (n_wd & 1) : ((n_wd >> 1) & 1));
      tc_fence_after();
      const uint32_t d = tmem_base + kDB + (uint32_t)(tb * 128);
      const uint64_t b0 = dWd + (uint64_t)((wslot * kWdGroupBytes) >> 4);
      if (elect_one()) {
#pragma unroll
        for (int kc = 0; kc < 2; ++kc)
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(d, a0 + (uint64_t)(kc * 1024 + k * 2), b0 + (uint64_t)(kc * 1024 + k * 2), idesc_b,
                      (uint32_t)((g | kc | k) != 0));
        umma_commit(&wd_empty[wslot]);
        if (HAS_TRAN) umma_commit(h_empty);
        else umma_commit(&empty_bar[s]);
        if (g == 3) umma_commit(&db_full[tb]);
      }
      __syncwarp();
      ++n_wd;
      if (HAS_TRAN) ++n_h;
      else if (++s == p.num_stages) { s = 0; phase ^= 1; }
      if (g == 3) { ++n_b[tb]; tb ^= kDBToggle; }
    };

    // HAS_TRAN: this thread issues phase A only; phase B has its own issuing thread (warp kFusedBWarp), so
    // that waiting for the converted tile / the weights never holds up the consumption of TMA stages.
    // tcgen05.commit tracks the MMAs of the issuing thread, so each thread signals exactly its own work.
    for (int tile = cta; tile < total_tiles; tile += ncta) {
      if (HAS_TRAN) {
        if (warp == 1) {
          for (int g = 0; g < 4; ++g) {
            if (MERGED) issue_u(g);
            issue_a(g);
          }
        } else {
          for (int g = 0; g < 4; ++g) issue_b(g);
        }
      } else {
        for (int g = 0; g < 4; ++g) issue_b(g);
      }
    }
    }
  } else if (MERGED && warp == kFusedWdWarp) {
    // ===================== LR-box + weight streamer (MERGED) =====================
    // slot 0 of the weight ring: the transposed-conv weights Wu_g (4 taps x [128 n][32 k], 64B swizzle), slot 1: the
    // conv weights Wd_g.  Wu of the next group is requested before Wd of this one: Wu_{g+1} only waits for the T_U
    // MMAs of group g, Wd_g for phase B of group g-1.  The LR boxes of a tile go with its Wu_0 (both wait for the last
    // T_U MMAs of the previous tile).
    uint32_t n_wu = 0, n_wdm = 0, n_lrl = 0;
    auto load_u = [&](int tile, int g) {
      if (g == 0) {
        int x0, y0, b;
        tile_coord(tile, x0, y0, b);
        mbar_wait(lr_empty, (n_lrl & 1) ^ 1);
        if (elect_one()) {
          // dx = -1 and dx = 0 boxes of 16 x 9 LR pixels; the dy = -1 / 0 taps are rows 0 and 1 of them
          mbar_expect_tx(lr_full, (uint32_t)kLRBytes);
          tma_load_4d(s_lr, &p.up_map, lr_full, 0, x0 - 1, y0 - 1, b);
          tma_load_4d(s_lr + kLRBox, &p.up_map, lr_full, 0, x0, y0 - 1, b);
        }
        __syncwarp();
        ++n_lrl;
      }
      mbar_wait(&wd_empty[0], (n_wu & 1) ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&wd_full[0], kWdGroupBytes);
        for (int t = 0; t < 4; ++t) tma_load_2d(s_wd + t * kWuTapBytes, &p.wu_map, &wd_full[0], t * 32, g * 128);
      }
      __syncwarp();
      ++n_wu;
    };
    if (cta < total_tiles) load_u(cta, 0);
    for (int tile = cta; tile < total_tiles; tile += ncta)
      for (int g = 0; g < 4; ++g) {
        if (g < 3) load_u(tile, g + 1);
        else if (tile + ncta < total_tiles) load_u(tile + ncta, 0);
        mbar_wait(&wd_empty[1], (n_wdm & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&wd_full[1], kWdGroupBytes);
          tma_load_2d(s_wd + kWdGroupBytes, &p.wd_map, &wd_full[1], (2 * g) * 64, 0);
          tma_load_2d(s_wd + kWdGroupBytes + 16384, &p.wd_map, &wd_full[1], (2 * g + 1) * 64, 0);
        }
        __syncwarp();
        ++n_wdm;
      }
  } else if (warp == kFusedWdWarp) {
    // ===================== conv-weight streamer =====================
    // every tile needs the 128 KB of 8x8-s4 weights once, 32 KB per sub-position group; all SMs
    // stream the same bytes, so these are L2 hits.  A 2-deep ring instead of a resident copy frees
    // 64 KB of shared memory for the activation pipeline (HBM latency hiding).
    uint32_t n_wd = 0;
    for (int tile = cta; tile < total_tiles; tile += ncta)
      for (int g = 0; g < 4; ++g) {
        const int slot = n_wd & 1;
        mbar_wait(&wd_empty[slot], ((n_wd >> 1) & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&wd_full[slot], kWdGroupBytes);
          tma_load_2d(s_wd + slot * kWdGroupBytes, &p.wd_map, &wd_full[slot], (2 * g) * 64, 0);
          tma_load_2d(s_wd + slot * kWdGroupBytes + 16384, &p.wd_map, &wd_full[slot], (2 * g + 1) * 64, 0);
        }
        __syncwarp();
        ++n_wd;
      }
  } else if (warp >= 2 && warp < 2 + kFusedEpiWarps) {
    // ===================== epilogue warps 2..17 =====================
    // warp -> TMEM lane quarter q = warp % 4 (hardware rule) and sub = which of the 4 column groups
    // (phase A: sub-position within the group; final: tap) this warp handles
    const int q = warp & 3;
    const int sub = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t m_a[2] = {0, 0}, m_b[2] = {0, 0}, m_h = 0;
    int tb = 0;
    const PreluCfg pc = make_prelu(HAS_TRAN ? s_bias[32] : 1.0f, 1);
    uint32_t m_u = 0;
    for (int tile = cta; tile < total_tiles; tile += ncta) {
      int x0, y0, b;
      tile_coord(tile, x0, y0, b);
      const int Yb = y0 + (row >> 4), Xb = x0 + (row & 15);
      const bool in_tensor = (Yb <= p.lr_h) && (Xb <= p.lr_w);
      if (HAS_TRAN) {
#pragma unroll 1
        for (int g = 0; g < 4; ++g) {
          const int buf = g & 1;
          if (MERGED) {
            // U_g = PReLU(T_U + b): sub-position s16 of this warp, zero ring as in igemm_kernel<EPI_DECONV>, written
            // into s_h in the layout of the two pair-plane TMA boxes -- phase A's operand for source nsrc-1 and, for
            // the groups whose hr map a later group reads, the source of two TMA stores into it
            mbar_wait_poll(tu_full, m_u & 1);
            tc_fence_after();
            uint32_t v[32];
            tmem_ld32(lane_base + kTU + (uint32_t)(sub * 32), v);
            tmem_ld_wait();
            tc_fence_before();
            mbar_arrive_warp(tu_empty);
            ++m_u;
            const int s16 = g * 4 + sub, ry = s16 >> 2, rx = s16 & 3;
            const int Yt = 4 * Yb + ry - 2, Xt = 4 * Xb + rx - 2;
            const bool inside = (Yt >= 0) && (Yt < 4 * p.lr_h) && (Xt >= 0) && (Xt < 4 * p.lr_w);
            uint32_t o[16];
            const PreluCfg pcu = make_prelu(s_ubias[32], 1);
            convert32(v, s_ubias, pcu, o);
            if (__builtin_expect(!inside, 0)) zero16(o);
            mbar_wait(h_empty, (m_h & 1) ^ 1);     // phase B of the previous group has read H from s_h
            uint8_t* urow = s_h + (sub >> 1) * 16384 + row * 128;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int piece = (sub & 1) * 4 + j;
              *reinterpret_cast<uint4*>(urow + ((piece ^ (row & 7)) << 4)) =
                  make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
            }
            fence_async_smem();
            asm volatile("bar.sync 1, %0;" ::"n"(32 * kFusedEpiWarps) : "memory");   // all of U_g is written
            if (threadIdx.x == 64) {   // one thread issues and later waits for the stores (bulk groups are per thread)
              if (p.hr_store) {
                tma_store_4d(&p.hr_maps[p.nsrc - 1], s_h, 0, x0, y0, b * 8 + 2 * g);
                tma_store_4d(&p.hr_maps[p.nsrc - 1], s_h + 16384, 0, x0, y0, b * 8 + 2 * g + 1);
                tma_store_commit();
              }
              mbar_arrive(u_full);
            }
          }
          mbar_wait_poll(&da_full[buf], m_a[buf] & 1);
          tc_fence_after();
          uint32_t o[16];
          uint32_t v[32];
          tmem_ld32(lane_base + (uint32_t)(buf * 128 + sub * 32), v);
          tmem_ld_wait();
          tc_fence_before();
          mbar_arrive_warp(&da_empty[buf]);
          const int s16 = g * 4 + sub, ry = s16 >> 2, rx = s16 & 3;
          const bool ring = (Yb == 0 && ry < 2) || (Yb == p.lr_h && ry >= 2) || (Xb == 0 && rx < 2) ||
                            (Xb == p.lr_w && rx >= 2);
          convert32(v, s_bias, pc, o);
          if (__builtin_expect(!(in_tensor && !ring), 0)) zero16(o);
          ++m_a[buf];
          if (MERGED) {
            // D_A is complete, so phase A has read U_g; the stores must have read it too before H overwrites it
            if (p.hr_store) {
              if (threadIdx.x == 64) tma_store_wait_read();
              asm volatile("bar.sync 1, %0;" ::"n"(32 * kFusedEpiWarps) : "memory");
            }
          } else {
            mbar_wait(h_empty, (m_h & 1) ^ 1);
          }
          // K index inside the group: k = sub*32 + c -> 64-element chunk kc = sub>>1, 16-byte piece (sub&1)*4 + j
          uint8_t* hrow = s_h + (sub >> 1) * 16384 + (row >> 3) * 1024 + (row & 7) * 128;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int piece = (sub & 1) * 4 + j;
            *reinterpret_cast<uint4*>(hrow + ((piece ^ (row & 7)) << 4)) =
                make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
          }
          fence_async_smem();
          mbar_arrive_warp(h_full);
          ++m_h;
        }
      }
      // final: channels [8*sub, 8*sub+8) of the four tap partials of D_B[tb].  Block (Yb,Xb)'s tap (dy,dx)
      // belongs to LR pixel (Yb-dy, Xb-dx).  The dx=1 partial is handed to the left neighbour lane (same block
      // row of the tile) by shuffle, giving each lane the two row partials comb[dy] of pixels (Yb-dy, Xb).
      //  * INTERIOR pixels -- tile rows 0..6, not the tile's last column: the second row partial is lane + 16's
      //    (lanes 0-15 hold block row 2q, lanes 16-31 block row 2q+1) or comes from the next lane quarter through a
      //    6 KB shared-memory exchange; the lane adds it to its comb[0], applies bias + PReLU and stores the
      //    finished BF16 pixel: 64 bytes instead of two FP32 slot writes, a finalize read of both and its store.
      //  * BOUNDARY pixels -- tile row 7 (its second partial lives in the next tile) and columns X % 16 == 15
      //    (their dx=1 partials live in the next tile), 18 % of the pixels: written, without atomics, to slots
      //    with exactly one writer each:  slot 2*dy   : tap (dy,0) + right neighbour's tap (dy,1)
      //                                   slot 2*dy+1 : tap (dy,1) arriving from the next tile
      //    finalize_lr_kernel sums them.  Same additions in the same order either way: deterministic.
      mbar_wait_poll(&db_full[tb], m_b[tb] & 1);
      tc_fence_after();
      uint32_t v[4][8];
#pragma unroll
      for (int t = 0; t < 4; ++t) tmem_ld8(lane_base + kDB + (uint32_t)(tb * 128 + t * 32 + sub * 8), v[t]);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive_warp(&db_empty[tb]);
      const int xl = lane & 15, half = lane >> 4;
      float comb[2][8];
#pragma unroll
      for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float right = __uint_as_float(v[dy * 2 + 1][k]);
          const float from_right = __shfl_down_sync(0xffffffffu, right, 1);
          comb[dy][k] = __uint_as_float(v[dy * 2][k]) + (xl < 15 ? from_right : 0.0f);
        }
      // second row partial of this lane's pixel (Yb, Xb): block row Yb+1's comb[1].  Even tile rows: lane + 16 of
      // this warp.  Odd tile rows 1, 3, 5: lanes 0-15 of the next lane quarter, through shared memory.
      float below[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) below[k] = __shfl_down_sync(0xffffffffu, comb[1][k], 16);
      if (half == 0 && q > 0) {
        float4* x = s_x + (((q - 1) * 4 + sub) * 16 + xl) * 2;
        x[0] = make_float4(comb[1][0], comb[1][1], comb[1][2], comb[1][3]);
        x[1] = make_float4(comb[1][4], comb[1][5], comb[1][6], comb[1][7]);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * kFusedEpiWarps) : "memory");     // the 16 epilogue warps only
      if (half == 1 && q < 3) {
        const float4* x = s_x + ((q * 4 + sub) * 16 + xl) * 2;
        const float4 x0v = x[0], x1v = x[1];
        below[0] = x0v.x; below[1] = x0v.y; below[2] = x0v.z; below[3] = x0v.w;
        below[4] = x1v.x; below[5] = x1v.y; below[6] = x1v.z; below[7] = x1v.w;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * kFusedEpiWarps) : "memory");     // reads done before the next tile's writes
      const int rr = 2 * q + half;                                               // block row inside the tile
      if (rr < 7 && xl < 15 && in_tensor && Yb < p.lr_h && Xb < p.lr_w) {   // interior pixel (Yb, Xb)
        const float slope = s_down[32];
        float r[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) r[k] = prelu(comb[0][k] + below[k] + s_down[sub * 8 + k], slope, 1);
        uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(p.lr_out) +
                                               ((((int64_t)b * p.lr_h + Yb) * p.lr_w + Xb) * 64 + sub * 16));
        *dst = make_uint4(pack_bf16(r[0], r[1]), pack_bf16(r[2], r[3]), pack_bf16(r[4], r[5]), pack_bf16(r[6], r[7]));
      }
#pragma unroll
      for (int dy = 0; dy < 2; ++dy) {
        const int Y = Yb - dy;
        if (in_tensor && Y >= 0 && Y < p.lr_h) {
          // row 7 of a tile, or the tile's last column
          const bool boundary = (((rr - dy) & 7) == 7) || (xl == 15);
          if (Xb < p.lr_w && boundary) {
            float4* dst = reinterpret_cast<float4*>(p.part + ((((int64_t)b * p.lr_h + Y) * p.lr_w + Xb) * 4 + 2 * dy) * 32 + sub * 8);
            dst[0] = make_float4(comb[dy][0], comb[dy][1], comb[dy][2], comb[dy][3]);
            dst[1] = make_float4(comb[dy][4], comb[dy][5], comb[dy][6], comb[dy][7]);
          }
          if (xl == 0 && Xb > 0) {
            float4* dst = reinterpret_cast<float4*>(p.part + ((((int64_t)b * p.lr_h + Y) * p.lr_w + Xb - 1) * 4 + 2 * dy + 1) * 32 + sub * 8);
            dst[0] = make_float4(__uint_as_float(v[dy * 2 + 1][0]), __uint_as_float(v[dy * 2 + 1][1]),
                                 __uint_as_float(v[dy * 2 + 1][2]), __uint_as_float(v[dy * 2 + 1][3]));
            dst[1] = make_float4(__uint_as_float(v[dy * 2 + 1][4]), __uint_as_float(v[dy * 2 + 1][5]),
                                 __uint_as_float(v[dy * 2 + 1][6]), __uint_as_float(v[dy * 2 + 1][7]));
          }
        }
      }
      ++m_b[tb];
      tb ^= kDBToggle;
    }
    if (MERGED && threadIdx.x == 64) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // the last stores
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<kTmemCols>(tmem_base);
  }
}

template <bool HAS_TRAN>
__global__ void __launch_bounds__(kFusedThreads, 1)
fused_down_kernel(const __grid_constant__ FusedDownParams p) {
  fused_down_body<HAS_TRAN, false>(p);
}

// One feedback group i >= 1 of the x4 stack with its transposed conv inside:
//
//     lr[i+1] = PReLU( Conv8x8s4( PReLU( Conv1x1( cat(hr[0..i-1], U_i) ) ) ) ),   U_i = PReLU( Deconv8x8s4(up_in) + b )
//
// U_i is made on chip one sub-position group g at a time, in the order phase A walks: the transposed conv's MMAs
// (T_U = LR taps * Wu_g^T, the 2 LR boxes of igemm_kernel<EPI_DECONV> loaded once per tile), the epilogue's conversion
// into s_h in the 128B-swizzled layout of the two pair-plane boxes phase A would load, two TMA stores of that buffer
// into hr[i] (only when a later group reads hr[i]: hr_store), and phase A's MMAs for source i from it.  Against the
// layered pair this removes the read of hr[i] (and for the last group its write) and the transposed conv's launch;
// the sums are the same additions in the same order, so the results are bit-identical.
//
// Resources (-Xptxas -v: 1 CTA per SM, no spills):
//  * TMEM, 512 columns: D_A double-buffered [0, 256), T_U [256, 384), D_B single [384, 512).  The epilogue is one
//    in-order sequence (U_g, H_g for g = 0..3, then the tile's D_B), so it always reads D_B before it produces the
//    next tile's first H and a second D_B buffer could never be used; a second D_A buffer lets phase A of group g+1
//    consume ring stages while the epilogue still reads D_A of group g.
//  * Weights: the 2 x 32 KB ring of the conv weights; slot 0 carries Wu_g (transposed conv, 32 KB per g), slot 1
//    Wd_g.  Both are L2 hits (every SM streams the same bytes).
//  * Shared memory: U_g and H_g share the 32 KB s_h (U_g is dead once D_A of g is complete and its stores have read
//    it; U_{g+1} waits for phase B of g); the LR boxes take 18 KB.  Activation ring: the deepest that fits, 6 x 16 KB
//    stages for nsrc 4, 5 for nsrc 5-6 (the layered kernel: 7 / 6); a ring one stage deeper does not fit, so the
//    comparison against one stage more is not measured.
__global__ void __launch_bounds__(kFusedThreads, 1)
fused_updown_kernel(const __grid_constant__ FusedDownParams p) {
  fused_down_body<true, true>(p);
}

// Boundary pixels (rows Y % 8 == 7 and columns X % 16 == 15; see the fused kernel's final epilogue):
// lr_out[p, c] = bf16(PReLU(sum of the pixel's partial slots + bias[c])).  8 channels per thread.
// Deterministic: every slot has one writer, the sum order is fixed.
constexpr int kFinalizePeriod = 8;   // boundary rows: one per 8-row tile
__global__ void __launch_bounds__(256)
finalize_lr_kernel(const float4* __restrict__ part, const float* __restrict__ bias, uint4* __restrict__ out, int B, int h,
                   int w) {
  // Work items = boundary pixels only, enumerated arithmetically (the first version walked every pixel and skipped
  // the interior ones): first the full rows Y = 8*k + 7, then, in the other rows, the columns X = 16*j + 15.
  constexpr int period = kFinalizePeriod;
  const float slope = __ldg(bias + 32);
  const int R = h / period, Cc = w / 16;
  const int64_t nA = (int64_t)B * R * w, nB = (int64_t)B * (h - R) * Cc;
  const int64_t n8 = (nA + nB) * 4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    const int c8 = (int)(i & 3);
    int64_t it = i >> 2;
    int b, Y, X;
    if (it < nA) {
      X = (int)(it % w);
      const int64_t r = it / w;
      Y = (int)(r % R) * period + period - 1;
      b = (int)(r / R);
    } else {
      it -= nA;
      X = (int)(it % Cc) * 16 + 15;
      const int64_t r = it / Cc;
      const int yy = (int)(r % (h - R));
      Y = yy + yy / (period - 1);
      b = (int)(r / (h - R));
    }
    const bool last_col = (X & 15) == 15;
    const int64_t px = ((int64_t)b * h + Y) * w + X;
    const float4* base = part + px * 32 + c8 * 2;          // 32 float4 per pixel, 8 per slot
    float4 a0 = base[0], a1 = base[1];
    const float4 b0 = base[16], b1 = base[17];
    a0 = make_float4(a0.x + b0.x, a0.y + b0.y, a0.z + b0.z, a0.w + b0.w);
    a1 = make_float4(a1.x + b1.x, a1.y + b1.y, a1.z + b1.z, a1.w + b1.w);
    if (last_col) {
      const float4 c0 = base[8], c1 = base[9], d0 = base[24], d1 = base[25];
      a0 = make_float4(a0.x + (c0.x + d0.x), a0.y + (c0.y + d0.y), a0.z + (c0.z + d0.z), a0.w + (c0.w + d0.w));
      a1 = make_float4(a1.x + (c1.x + d1.x), a1.y + (c1.y + d1.y), a1.z + (c1.z + d1.z), a1.w + (c1.w + d1.w));
    }
    float r[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = prelu(r[k] + __ldg(bias + c8 * 8 + k), slope, 1);
    out[px * 4 + c8] = make_uint4(pack_bf16(r[0], r[1]), pack_bf16(r[2], r[3]), pack_bf16(r[4], r[5]), pack_bf16(r[6], r[7]));
  }
}

}  // namespace vsr
