// projection.cu -- forward flow projection (a1) and inverse-depth-weighted projection (a2):
// splat with accumulation + count, normalise, hole mask, 4-direction hole fill.
//
// Contract: SURVEY.md Appendix B (the reference ships only the Module surfaces,
// FlowProjectionModule.py:18-33 / DepthProjectionModule.py:12-18; the splat itself has no
// reference implementation -- parity unpinned, oracle/oracle.c::or_flow_projection is the spec).
//
// The four targets of a source pixel all receive the SAME value (Appendix B step 2: no bilinear weights), so the
// splat factors into (1) a histogram over CELLS -- every source adds {-fx*D, -fy*D, D, 1} once to cell
// (int(y2), int(x2)) -- and (2) a 2x2 box sum: target (ty,tx) = cell(ty,tx) + cell(ty,tx-1) + cell(ty-1,tx) +
// cell(ty-1,tx-1), the clamped duplicates of the last row / column being a multiplicity 2.  A cell is one float4;
// the count rides along as a float (exact below 2^24) and is exported as int32 -> count / hole bit-exact.
//
// Two paths:
//  * BOUNDED displacement (caller promises |fx|,|fy| <= max_disp <= 8 px; the pipeline's smooth +-8 px fields):
//    owner-computes in shared memory.  A CTA owns a 128x80 target tile; its 129x81 cells live in shared memory.  The
//    sources that can reach them (tile +- 8, 1.5 candidates per target) are cut into 16x16 blocks; blocks whose origins
//    differ by 32 can never touch the same cell, so the blocks are processed in 4 colour phases, one warp per block,
//    with plain LDS/STS read-modify-writes -- no atomics; lanes of one instruction that hit the same cell are
//    serialised by a one-byte claim protocol.  Box sum + normalise + masks + bitmaps then stream out of shared memory
//    in one coalesced pass that also lists the row words with holes for the fill.  No global accumulator, no memset,
//    no second pass over the cells: HBM sees the algorithmic bytes only.  A source that breaks the promise raises a
//    flag and the whole batch is redone by the general path (one gated launch that exits at once otherwise).
//  * GENERAL (config C3's +-64 px): scatter with one 16-byte red.global.add.v4.f32 per source into ONE L2-resident
//    cell array (33 MB at 1080p), then a gather pass (box sum + normalise + masks + the list of row words with holes)
//    and the fill over that list (which also clears the cell array for the next image), image after image on the
//    caller's stream.  Overlapping the stages of successive images was tried three ways and measured slower (see
//    run_general); the cooperative pipelined kernel of those experiments survives as the gated fallback of the
//    bounded path, where what matters is that skipping it costs one empty launch.
#include <cooperative_groups.h>


#include "common.cuh"

namespace cg = cooperative_groups;

namespace vsr {
namespace {

constexpr int kThreads = 256;
constexpr int kRows = 8;  // rows walked by one splat warp task (all of their flow / depth loads are issued up front)

// Reads of data another CTA wrote earlier in the SAME (persistent) kernel go to L2 (ld.global.cg): the non-coherent
// path of __ldg / const __restrict__ may serve a line this SM cached from the previous use of a rotating buffer.
template <bool CG> __device__ __forceinline__ float4 ldg_f4(const float4* p) { return CG ? __ldcg(p) : __ldg(p); }
__device__ __forceinline__ float4 shfl_up1_f4(float4 v) {
  return make_float4(__shfl_up_sync(0xffffffffu, v.x, 1), __shfl_up_sync(0xffffffffu, v.y, 1),
                     __shfl_up_sync(0xffffffffu, v.z, 1), __shfl_up_sync(0xffffffffu, v.w, 1));
}
__device__ __forceinline__ void red_add_f4(float4* addr, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

// Everything the kernels need to find the buffers of image b.
struct ProjArgs {
  const float* flow;       // (B,h,w,2)
  const float* inv_depth;  // (B,h,w) or nullptr
  float* proj;             // (B,h,w,2)
  float* wsum;             // (B,h,w) or nullptr
  int32_t* count;          // (B,h,w)
  uint8_t* hole;           // (B,h,w)
  float4* acc;             // 3 cell arrays of h*w float4 (general path)
  uint32_t* rowmask;       // per image: h * ceil(w/32) words, bit x%32 of word (y, x/32) = pixel has hits
  uint32_t* colmask;       // per image: ceil(h/32) * w words, bit y%32 of word (y/32, x)
  int* flags;              // [0] promise broken (bounded path), [1 + b] image b has holes, [1 + B] length of holelist
  uint32_t* holelist;      // bounded path: the row words (b * h * ceil(w/32) + word) that contain holes
  int B, h, w;
  int gate;                // general path: 1 = run only if flags[0] != 0 (fallback of the bounded path)
};

__device__ __forceinline__ int64_t rowmask_words(int h, int w) { return (int64_t)h * ceil_div(w, 32); }
__device__ __forceinline__ int64_t colmask_words(int h, int w) { return (int64_t)ceil_div(h, 32) * w; }

// Normalisation of one target from its box sum a = {sum -fx*D, sum -fy*D, sum D, count}.  A target is a hole when
// nothing hit it, and also when the hits carry no usable weight (sum D <= 0 or NaN: an inverse depth of 0 from a
// real estimator) -- dividing by it would put NaN into the warp and the whole conv stack.
__device__ __forceinline__ bool normalise_target(const float4 a, float2& o) {
  const bool is_hole = !(a.w > 0.0f) || !(a.z > 0.0f);
  o = make_float2(0.f, 0.f);
  if (!is_hole) {
    float rz;                            // one approximate reciprocal (1 ulp), two products: ~2 ulp from the quotients,
    asm("rcp.approx.f32 %0, %1;" : "=f"(rz) : "f"(a.z));   // far inside the 1e-3 contract; no slow path
    o = make_float2(a.x * rz, a.y * rz);
  }
  return is_hole;
}

// The same with a single MUFU for the reciprocal: rcp.approx.ftz is exact to 1 ulp for normal operands; the (never
// seen) denormal or > 2^126 weight sums take the full division.
__device__ __forceinline__ bool normalise_target_fast(const float4 a, float2& o) {
  const bool is_hole = !(a.w > 0.0f) || !(a.z > 0.0f);
  o = make_float2(0.f, 0.f);
  if (!is_hole) {
    if (a.z >= 1.17549435e-38f && a.z <= 8.5e37f) {
      float rz;
      asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rz) : "f"(a.z));
      o = make_float2(a.x * rz, a.y * rz);
    } else {
      float2 q;
      normalise_target(a, q);
      o = q;
    }
  }
  return is_hole;
}

// ---------------------------------------------------------------------------------------------
// GENERAL path, stage roles.  Each role spreads its work over `nw` warps (the whole grid) by a warp-stride loop.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void role_zero(float4* __restrict__ acc, int64_t n, int64_t tid, int64_t nthreads) {
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t i = tid; i < n; i += nthreads) acc[i] = z;
}

// One warp task = 32 consecutive x, kRows consecutive rows.
__device__ __forceinline__ void role_splat(const float* __restrict__ flow, const float* __restrict__ inv_depth,
                                           float4* __restrict__ acc, int h, int w, int warp0, int nw, int lane) {
  const int warps_x = ceil_div(w, 32);
  const int n_tasks = warps_x * ceil_div(h, kRows);
  const float xmax = (float)(w - 1), ymax = (float)(h - 1);
  for (int task = warp0; task < n_tasks; task += nw) {
    const int x = (task % warps_x) * 32 + lane;
    const int y0 = (task / warps_x) * kRows;
    // ncu (first version): 48 % of the stall samples sat on the first use of the flow load -- a warp
    // walked its rows with one dependent load per row.  Issue every row's loads first.
    float2 fl[kRows];
    float dp[kRows];
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
      const int y = y0 + r;
      fl[r] = make_float2(0.f, 0.f);
      dp[r] = 1.0f;
      if (x < w && y < h) {
        const int64_t p = (int64_t)y * w + x;
        fl[r] = ldg_stream_f2(reinterpret_cast<const float2*>(flow) + p);
        if (inv_depth) dp[r] = __ldg(inv_depth + p);
      }
    }
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
      const int y = y0 + r;
      if (x < w && y < h) {
        const float2 f = fl[r];
        const float x2 = __fadd_rn((float)x, f.x);
        const float y2 = __fadd_rn((float)y, f.y);
        // Appendix B step 2 (the comparison form also rejects NaN)
        if (x2 >= 0.0f && x2 <= xmax && y2 >= 0.0f && y2 <= ymax) {
          const float d = dp[r];
          red_add_f4(acc + ((int)y2 * w + (int)x2), make_float4(__fmul_rn(-f.x, d), __fmul_rn(-f.y, d), d, 1.0f));
        }
      }
    }
  }
}

// 2x2 box sum of the cells + normalise + hole mask, and the occupancy bitmaps the fill uses.  One warp task = one
// 32-wide, kStrip-tall strip: lane = column, the warp walks the rows.  The cell above is the previous row's own cell (a
// register), the cells to the left come from the neighbouring lane by shuffle (lane 0 loads them), so every cell is
// loaded once; 4 rows of loads are in flight at a time.  The ballot of "has hits" is the row word; each lane collects
// its own column bits and writes its byte of the column word -- no shared memory, no block barrier.  Hole pixels
// get (0,0) here; the fill overwrites them.  The row words with holes go on a list for the fill.
constexpr int kStrip = 8, kBatch = 4;      // 8 rows per warp task: twice the warps of 16-row strips for the same loads in flight

template <bool CG, bool LOOP>
__device__ __forceinline__ void role_normalise(const float4* __restrict__ acc, float* __restrict__ proj,
                                               float* __restrict__ wsum, int32_t* __restrict__ count,
                                               uint8_t* __restrict__ hole, uint32_t* __restrict__ rowmask,
                                               uint32_t* __restrict__ colmask, int* __restrict__ has_holes,
                                               uint32_t* __restrict__ holelist, int h, int w, int warp0, int nw, int lane) {
  // holelist != nullptr: *has_holes counts the row words with holes and holelist names them (the fill then visits only
  // those); nullptr: *has_holes is a flag and the fill scans every word
  const int tiles_x = ceil_div(w, 32);
  const int n_strips = (32 / kStrip) * ceil_div(h, 32);   // every byte of every column word gets written
  const int n_tasks = tiles_x * n_strips;
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  // LOOP = false: the stand-alone launch gives every warp exactly one strip (the loop's live range costs the 64-register
  // kernel spills in its inner loop)
  for (int task = warp0; task < n_tasks; task += LOOP ? nw : n_tasks) {
    const int tx = task % tiles_x, strip = task / tiles_x;
    const int x = tx * 32 + lane, y0 = strip * kStrip;
    const bool in_x = x < w;
    const float mx = (x == w - 1) ? 2.0f : 1.0f;
    float4 up = (in_x && y0 > 0 && y0 <= h) ? ldg_f4<CG>(acc + (y0 - 1) * w + x) : zero4;            // cell (y0-1, x)
    float4 up_left = shfl_up1_f4(up);                                                              // cell (y0-1, x-1)
    if (lane == 0) up_left = (x > 0 && y0 > 0 && y0 <= h) ? ldg_f4<CG>(acc + (y0 - 1) * w + x - 1) : zero4;
    uint32_t colbits = 0;
    uint32_t holerows = 0;                             // warp-uniform: rows of the strip whose word has a hole
    const uint32_t inx_mask = __ballot_sync(0xffffffffu, in_x);
#pragma unroll
    for (int r0 = 0; r0 < kStrip; r0 += kBatch) {
      float4 c[kBatch], cl[kBatch];
#pragma unroll
      for (int r = 0; r < kBatch; ++r) {
        const int y = y0 + r0 + r;
        c[r] = (in_x && y < h) ? ldg_f4<CG>(acc + y * w + x) : zero4;
        cl[r] = (lane == 0 && x > 0 && y < h) ? ldg_f4<CG>(acc + y * w + x - 1) : zero4;
      }
#pragma unroll
      for (int r = 0; r < kBatch; ++r) {
        const int y = y0 + r0 + r;
        const float4 c11 = c[r], c01 = up;
        float4 c10 = shfl_up1_f4(c11);
        if (lane == 0) c10 = cl[r];
        const float4 c00 = up_left;            // cell (y-1, x-1) = the previous row's left neighbour
        up = c11;
        up_left = c10;
        const bool in_img = in_x && y < h;
        bool is_hole = false;
        if (in_img) {
          // 2x2 box sum in a fixed order; the clamped duplicate targets (Appendix B: "hit twice") are the
          // multiplicity 2 of the target's own column at x = w-1 and of its own row at y = h-1
          const float my = (y == h - 1) ? 2.0f : 1.0f;
          float4 a;
          a.x = (c11.x * mx + c10.x) * my + (c01.x * mx + c00.x);
          a.y = (c11.y * mx + c10.y) * my + (c01.y * mx + c00.y);
          a.z = (c11.z * mx + c10.z) * my + (c01.z * mx + c00.z);
          a.w = (c11.w * mx + c10.w) * my + (c01.w * mx + c00.w);
          const int p = y * w + x;
          float2 o;
          is_hole = normalise_target(a, o);
          reinterpret_cast<float2*>(proj)[p] = o;
          if (wsum) wsum[p] = is_hole ? 0.0f : a.z;
          count[p] = (int32_t)a.w;
          hole[p] = is_hole ? 1 : 0;
        }
        const uint32_t m = __ballot_sync(0xffffffffu, in_img && !is_hole);
        if (lane == 0 && y < h) rowmask[y * tiles_x + tx] = m;
        colbits |= (uint32_t)(in_img && !is_hole) << (r0 + r);
        holerows |= (uint32_t)(y < h && (inx_mask & ~m) != 0) << (r0 + r);
      }
    }
    if (in_x) reinterpret_cast<uint8_t*>(colmask)[((strip >> 2) * w + x) * 4 + (strip & 3)] = (uint8_t)colbits;
    if (holerows) {
      if (holelist) {
        const int nh = __popc(holerows);
        int base = 0;
        if (lane == 0) base = atomicAdd(has_holes, nh);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (lane < nh) holelist[base + lane] = (uint32_t)((y0 + __fns(holerows, 0, lane + 1)) * tiles_x + tx);
      } else if (lane == 0) {
        *reinterpret_cast<volatile int*>(has_holes) = 1;   // a flag, not a count: plain store
      }
    }
  }
}

// 4-direction fill (Appendix B step 4): nearest pixel with hits to the left, right, up and down; mean of the found
// (1-4) normalised values, summed in that order; (0,0) if none.  The searches run on the bitmaps, 32 pixels per step.
// One warp per 32-pixel row word: a word without holes costs one 4-byte load for the whole warp; the hole pixels of a
// word are filled in parallel by their lanes.  Only non-hole pixels are read, so the result does not depend on
// execution order.
template <bool CG>
__device__ __forceinline__ void fill_word(const uint32_t* rowmask_, const uint32_t* colmask_, float* proj, int h, int w,
                                          int wd, int lane) {
  struct Words { const uint32_t* p; __device__ __forceinline__ uint32_t operator[](int64_t i) const { return CG ? __ldcg(p + i) : __ldg(p + i); } };
  const Words rowmask{rowmask_}, colmask{colmask_};
  const int wpr = ceil_div(w, 32), hpr = ceil_div(h, 32);
  const float2* pin = reinterpret_cast<const float2*>(proj);   // non-hole pixels only: never written here
  const int y = wd / wpr, seg0 = wd - y * wpr;
  const int x = seg0 * 32 + lane;
  const uint32_t hits = rowmask[wd];
  if (x >= w || ((hits >> lane) & 1u)) return;
  const int p = y * w + x;
  // the four searches first (bitmap words only), then the four neighbour values in flight together, summed in the
  // order left, right, up, down
  int nx[4], ny[4];
  bool has[4] = {false, false, false, false};
  {  // left
    int seg = x >> 5;
    uint32_t word = hits & ((1u << (x & 31)) - 1u);
    while (word == 0 && seg > 0) word = rowmask[y * wpr + --seg];
    has[0] = word != 0;
    nx[0] = seg * 32 + 31 - __clz(word);
    ny[0] = y;
  }
  {  // right
    int seg = x >> 5;
    uint32_t word = hits & ~((2u << (x & 31)) - 1u);
    while (word == 0 && seg + 1 < wpr) word = rowmask[y * wpr + ++seg];
    has[1] = word != 0;
    nx[1] = seg * 32 + __ffs(word) - 1;
    ny[1] = y;
  }
  const uint32_t cword = colmask[(y >> 5) * w + x];
  {  // up
    int sb = y >> 5;
    uint32_t word = cword & ((1u << (y & 31)) - 1u);
    while (word == 0 && sb > 0) word = colmask[--sb * w + x];
    has[2] = word != 0;
    nx[2] = x;
    ny[2] = sb * 32 + 31 - __clz(word);
  }
  {  // down
    int sb = y >> 5;
    uint32_t word = cword & ~((2u << (y & 31)) - 1u);
    while (word == 0 && sb + 1 < hpr) word = colmask[++sb * w + x];
    has[3] = word != 0;
    nx[3] = x;
    ny[3] = sb * 32 + __ffs(word) - 1;
  }
  float2 q[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {     // the neighbours' normalised values, as written by the normalise pass
    q[k] = make_float2(0.f, 0.f);
    if (has[k]) q[k] = CG ? __ldcg(pin + ny[k] * w + nx[k]) : pin[ny[k] * w + nx[k]];
  }
  float sx = 0.f, sy = 0.f;
  int found = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (has[k]) {
      sx += q[k].x;
      sy += q[k].y;
      ++found;
    }
  if (found > 0) reinterpret_cast<float2*>(proj)[p] = make_float2(__fdiv_rn(sx, (float)found), __fdiv_rn(sy, (float)found));
}

template <bool CG>
__device__ __forceinline__ void role_fill(const uint32_t* rowmask, const uint32_t* colmask, float* proj, int h, int w,
                                          int warp0, int nw, int lane) {
  const int n_words = h * ceil_div(w, 32);
  for (int wd = warp0; wd < n_words; wd += nw) fill_word<CG>(rowmask, colmask, proj, h, w, wd, lane);
}

// The general path: one cooperative persistent kernel over the whole batch.  Phase p (p = -1 .. B+1):
//   zero the cell array of image p+1 | splat image p | normalise image p-1 | fill image p-2, then a grid barrier.
// Every CTA does its slice of every role; CTAs start at different roles so that at any moment the chip runs a mix of
// the four (the reduction issue rate bounds the splat, L2 reads + HBM writes the normalise, latency the fill).
__global__ void __launch_bounds__(kThreads, 3)
projection_pipeline_kernel(const ProjArgs a) {
  if (a.gate && *reinterpret_cast<volatile int*>(a.flags) == 0) return;   // uniform: nobody reaches a barrier
  cg::grid_group grid = cg::this_grid();
  const int lane = threadIdx.x & 31;
  const int nw = (gridDim.x * kThreads) >> 5;
  const int warp0 = (blockIdx.x * kThreads + threadIdx.x) >> 5;
  const int64_t tid = (int64_t)blockIdx.x * kThreads + threadIdx.x, nthreads = (int64_t)gridDim.x * kThreads;
  const int64_t P = (int64_t)a.h * a.w;
  const int64_t rw = rowmask_words(a.h, a.w), cw = colmask_words(a.h, a.w);
  for (int p = -1; p <= a.B + 1; ++p) {
    if (p == -1)
      for (int64_t i = tid; i < a.B; i += nthreads) a.flags[1 + i] = 0;
#pragma unroll 1
    for (int k = 0; k < 4; ++k) {
      const int role = (k + blockIdx.x) & 3;
      if (role == 0) {
        if (p + 1 < a.B) role_zero(a.acc + ((p + 1) % 3) * P, P, tid, nthreads);
      } else if (role == 1) {
        if (p >= 0 && p < a.B)
          role_splat(a.flow + p * P * 2, a.inv_depth ? a.inv_depth + p * P : nullptr, a.acc + (p % 3) * P, a.h, a.w,
                     warp0, nw, lane);
      } else if (role == 2) {
        const int b = p - 1;
        if (b >= 0 && b < a.B)
          role_normalise<true, true>(a.acc + (b % 3) * P, a.proj + b * P * 2, a.wsum ? a.wsum + b * P : nullptr, a.count + b * P,
                         a.hole + b * P, a.rowmask + b * rw, a.colmask + b * cw, a.flags + 1 + b, nullptr, a.h, a.w,
                         warp0, nw, lane);
      } else {
        const int b = p - 2;
        if (b >= 0 && b < a.B && *reinterpret_cast<volatile int*>(a.flags + 1 + b) != 0)
          role_fill<true>(a.rowmask + b * rw, a.colmask + b * cw, a.proj + b * P * 2, a.h, a.w, warp0, nw, lane);
      }
    }
    if (p <= a.B) grid.sync();
  }
}

// The stage kernels of the general path are short (5-15 us) and strictly dependent, so their launch gaps count: they
// are launched with programmatic stream serialization -- the next stage's CTAs may become resident while the last CTAs
// of this one drain -- and every stage starts by letting its successor launch and then waiting for its predecessor to
// have completed and flushed (griddepcontrol.wait).  (The layers of the conv stack, 0.1-2 ms each, measured no gain
// from this: DESIGN.md section 6.)
__device__ __forceinline__ void chain_enter() {
  griddep_launch_dependents();
  griddep_wait();
}
template <typename... KArgs, typename... Args>
inline int launch_chained(void (*kernel)(KArgs...), int grid, int block, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid, 1, 1);
  cfg.blockDim = dim3((unsigned)block, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
  if (e != cudaSuccess) return cuda_status(e);
  return after_launch();
}

// The same stages as stand-alone kernels, each with its own register budget / occupancy (the merged kernel above runs
// every role at 24 warps per SM; alone the splat keeps 64 in flight): the general path (run_general).
__global__ void __launch_bounds__(kThreads)
stage_splat_kernel(const float* __restrict__ flow, const float* __restrict__ inv_depth, float4* __restrict__ acc, int h, int w) {
  chain_enter();
  role_splat(flow, inv_depth, acc, h, w, (blockIdx.x * kThreads + threadIdx.x) >> 5, (gridDim.x * kThreads) >> 5, threadIdx.x & 31);
}
__global__ void __launch_bounds__(kThreads, 4)
stage_normalise_kernel(const float4* __restrict__ acc, float* __restrict__ proj, float* __restrict__ wsum,
                       int32_t* __restrict__ count, uint8_t* __restrict__ hole, uint32_t* __restrict__ rowmask,
                       uint32_t* __restrict__ colmask, int* __restrict__ n_holewords, uint32_t* __restrict__ holelist, int h,
                       int w) {
  chain_enter();
  role_normalise<false, false>(acc, proj, wsum, count, hole, rowmask, colmask, n_holewords, holelist, h, w,
                               (blockIdx.x * kThreads + threadIdx.x) >> 5, (gridDim.x * kThreads) >> 5, threadIdx.x & 31);
}
// fill of the general path: the row words of one image that the normalise stage listed
__global__ void __launch_bounds__(kThreads)
stage_fill_kernel(const uint32_t* rowmask, const uint32_t* colmask, const int* n_holewords, const uint32_t* holelist,
                  float* proj, float4* zero_acc, int h, int w) {
  chain_enter();
  // the cell array is free once the normalise stage is through: cleared here for the next image (one launch and its gap
  // less than a memset per image)
  if (zero_acc) role_zero(zero_acc, (int64_t)h * w, (int64_t)blockIdx.x * kThreads + threadIdx.x, (int64_t)gridDim.x * kThreads);
  const int n = *reinterpret_cast<const volatile int*>(n_holewords);
  const int nw = (gridDim.x * kThreads) >> 5, lane = threadIdx.x & 31;
  for (int i = (blockIdx.x * kThreads + threadIdx.x) >> 5; i < n; i += nw)
    fill_word<false>(rowmask, colmask, proj, h, w, (int)__ldg(holelist + i), lane);
}

// ---------------------------------------------------------------------------------------------
// BOUNDED path: owner-computes tiles in shared memory, 4-colour block phases.
// ---------------------------------------------------------------------------------------------
// Geometry (all for a displacement bound of kBD = 8 px; a smaller promise runs on the same geometry):
//  * a CTA owns a kTW x kTH target tile = (kTW+1) x (kTH+1) cells (the box sum needs the cell column to the left and
//    the cell row above); cells are float4 in shared memory;
//  * the sources that can reach those cells lie in [tx0-1-kBD, tx0+kTW-1+kBD] x [ty0-1-kBD, ty0+kTH-1+kBD].  That
//    region (x widened to 16-pixel alignment: 128-byte aligned flow rows) is cut into blocks of kBS x kBS = 16 x 16
//    sources.  A block's sources reach at most the 32 x 32 cells around it, so two blocks whose origins differ by a
//    multiple of 32 in x and y never touch the same cell: blocks are processed in 4 colour phases (x parity, y parity),
//    one warp per 2x2 super-block, a block barrier between the phases -> within a phase every cell is touched by
//    one warp only, plain LDS / STS read-modify-write, no atomics.  Candidates scanned per target: 1.5 (the previous
//    scheme -- a warp owns a cell rectangle and scans rectangle +- bound -- scanned 2.3 and needed ~100
//    instructions per 32 candidates);
//  * the last source row (ty0+kTH-1+kBD: it reaches the tile only with fy == -kBD exactly) does not fill a block row;
//    warp 15 walks it during the first phase, when no block that reaches cell row kTH is active;
//  * inside a warp, sources of one instruction that hit the same cell take turns through a one-byte claim protocol.
//    A lane holds 2 x 4 sources of its block (a column pair x 4 rows, one 16-byte flow load per row) and the rounds
//    are arranged so that the 64 sources of a round are 2 apart in x and in y: smooth fields (|gradient| < 0.5)
//    practically never collide, and the 8 lanes of a quarter warp hit 8 different 16-byte bank groups.
constexpr int kBD = 8;                              // displacement bound of the geometry
constexpr int kBS = 2 * kBD;                        // block side
constexpr int kTW = 128, kTH = 80;                  // target tile
constexpr int kCW = kTW + 1, kCH = kTH + 1;         // cells of a tile
constexpr int kNC = kCW * kCH;                      // 10 449 cells = 167 184 B
constexpr int kClaimPitch = 136;                    // claim bytes per cell row: rows 4 apart land 8 banks apart
constexpr int kSX0 = -16, kSY0 = -(kBD + 1);        // origin of the scanned source region relative to (tx0, ty0)
constexpr int kNBX = (kTW + 32) / kBS;              // 10 block columns: x in [tx0-16, tx0+144)
constexpr int kNBY = (kTH + kBS) / kBS;             // 6 block rows: y in [ty0-9, ty0+87), + the extra row ty0+87
static_assert(kNBX % 2 == 0 && kNBY % 2 == 0, "2x2 super-blocks");
static_assert(kSX0 <= -1 - kBD && kSX0 + kNBX * kBS > kTW - 1 + kBD, "x coverage");
static_assert(kSY0 + kNBY * kBS == kTH - 1 + kBD, "the extra row is the one after the last block row");
static_assert(kTH % 16 == 0 && kTW % 32 == 0, "bitmap granularity");
constexpr int kAccWarps = (kNBX / 2) * (kNBY / 2);  // 15 super-blocks
constexpr int kTileWarps = 16;
constexpr int kTileThreads = 32 * kTileWarps;
static_assert(kAccWarps < kTileWarps && kTileWarps % 4 == 0 && kTH % (kTileWarps / 4) == 0, "warp roles");
constexpr int kOutRows = kTH / (kTileWarps / 4);    // 20 target rows per output warp (4 column chunks of 32)
constexpr int kSeamRows = kTH / kOutRows + 1;       // cell rows 0, kOutRows, 2 kOutRows, ..: read by two output warps
constexpr int kSeamCells = kSeamRows * kCW + kCH * (kTW / 32 + 1);   // + cell columns 0, 32, 64, .. (all rows)
constexpr int kColWords = 4;                        // staged column bitmap: bit (ty0 % 32) + row, up to 16 + 79
constexpr int kMaxBound = kBD;
constexpr int kExtraChunks = kNBX * kBS / 32;       // the extra source row, 32 sources at a time
constexpr size_t kTileSmem = (size_t)(kNC + 32) * 16 + (size_t)kColWords * kTW * 4 + (size_t)kClaimPitch * kCH + 32;   // + scratch

struct TileRect {      // the tile's cells as bounds on the target position (x2, y2), and the tile's first cell
  float xa, xb, ya, yb;
  float cx0f, cy0f;
};

// One claim round for two sources per lane, as one block of PTX on 32-bit shared addresses (the compiler's version
// of the same logic rebuilt the shared window base and converted predicates to integers and back in every round).
// pend0/pend1 (in/out, 0 or 1): the source still has to be added.  Everybody pending writes its id to the claim byte
// of its cell, the survivor of a cell reads the cell, adds {vx, vy, d, 1} and writes it back, and stops pending.
// Branch-free; the loads are unpredicated (a predicated shared load into registers that are live afterwards costs
// ptxas a copy per register): a lane with nothing to add reads its OWN scratch cell / claim byte (scr_cell, scr_claim:
// one per lane, so idle lanes do not pile up on one bank as they did on a shared dummy cell); the stores are predicated.
// claim0/claim1 must already point at the scratch byte for sources that are not pending.
__device__ __forceinline__ void claim_round2(uint32_t& pend0, uint32_t& pend1, uint32_t& claim0, uint32_t& claim1,
                                             uint32_t id0, uint32_t id1, uint32_t cell0, uint32_t cell1, float vx0,
                                             float vy0, float d0, float vx1, float vy1, float d1, uint32_t scr_cell,
                                             uint32_t scr_claim) {
  asm volatile(
      "{\n"
      " .reg .pred w0, w1, p0, p1;\n"
      " .reg .b32 who0, who1, c0, c1;\n"
      " .reg .f32 a0, a1, a2, a3, b0, b1, b2, b3;\n"
      " setp.ne.u32 p0, %0, 0;\n"
      " setp.ne.u32 p1, %1, 0;\n"
      " @p0 st.shared.u8 [%2], %4;\n"
      " @p1 st.shared.u8 [%3], %5;\n"
      " bar.warp.sync 0xffffffff;\n"
      " ld.shared.u8 who0, [%2];\n"
      " ld.shared.u8 who1, [%3];\n"
      " setp.eq.u32 w0, who0, %4;\n"
      " setp.eq.u32 w1, who1, %5;\n"
      " and.pred w0, w0, p0;\n"
      " and.pred w1, w1, p1;\n"
      " selp.u32 c0, %6, %14, w0;\n"
      " selp.u32 c1, %7, %14, w1;\n"
      " ld.shared.v4.f32 {a0, a1, a2, a3}, [c0];\n"
      " ld.shared.v4.f32 {b0, b1, b2, b3}, [c1];\n"
      " add.f32 a0, a0, %8;\n"
      " add.f32 a1, a1, %9;\n"
      " add.f32 a2, a2, %10;\n"
      " add.f32 a3, a3, 0f3F800000;\n"
      " add.f32 b0, b0, %11;\n"
      " add.f32 b1, b1, %12;\n"
      " add.f32 b2, b2, %13;\n"
      " add.f32 b3, b3, 0f3F800000;\n"
      " @w0 st.shared.v4.f32 [c0], {a0, a1, a2, a3};\n"
      " @w1 st.shared.v4.f32 [c1], {b0, b1, b2, b3};\n"
      " selp.u32 %0, 0, %0, w0;\n"          // a winner is done: from now on it only touches its scratch byte (a winner
      " selp.u32 %1, 0, %1, w1;\n"          // that kept writing its id to the real claim byte would starve the others)
      " selp.u32 %2, %15, %2, w0;\n"
      " selp.u32 %3, %15, %3, w1;\n"
      " bar.warp.sync 0xffffffff;\n"
      "}\n"
      : "+r"(pend0), "+r"(pend1), "+r"(claim0), "+r"(claim1)
      : "r"(id0), "r"(id1), "r"(cell0), "r"(cell1), "f"(vx0), "f"(vy0), "f"(d0), "f"(vx1), "f"(vy1), "f"(d1),
        "r"(scr_cell), "r"(scr_claim)
      : "memory");
}

// Adds U (1 or 2) x 32 sources (flow fx/fy, inverse depth dd, position xs/ys; NaN flow = no source) to the tile's
// cells.  Sources of one call that hit the same cell take turns (claim_round2).
template <int U, bool VMAX>
__device__ __forceinline__ void add_sources(const float (&fx)[U], const float (&fy)[U], const float (&dd)[U],
                                            const float (&xs)[U], const float (&ys)[U], uint32_t cells_sa,
                                            uint32_t claim_sa, const TileRect& R, int lane, float& vmax) {
  static_assert(U == 1 || U == 2, "claim_round2");
  const uint32_t scr_cell = cells_sa + 16u * (uint32_t)(kNC + lane), scr_claim = claim_sa + (uint32_t)(kClaimPitch * kCH + lane);
  uint32_t cell_a[2] = {scr_cell, scr_cell}, claim_a[2] = {scr_claim, scr_claim}, pend[2] = {0, 0};
  float vx[2] = {0.f, 0.f}, vy[2] = {0.f, 0.f}, dv[2] = {0.f, 0.f};
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const float x2 = __fadd_rn(xs[u], fx[u]), y2 = __fadd_rn(ys[u], fy[u]);
    if (VMAX) vmax = fmaxf(vmax, fmaxf(fabsf(fx[u]), fabsf(fy[u])));
    // "lands in one of the tile's cells and inside the image" (Appendix B step 2; NaN fails every compare)
    const bool in = x2 >= R.xa && x2 <= R.xb && y2 >= R.ya && y2 <= R.yb;
    pend[u] = in ? 1u : 0u;
    // local cell: x2 - cx0 is exact (an integer below 2^11 off a float below 2^24) and >= 0 where it matters
    const int ix = (int)(x2 - R.cx0f), iy = (int)(y2 - R.cy0f);
    cell_a[u] = cells_sa + 16u * (uint32_t)(iy * kCW + ix);
    claim_a[u] = in ? claim_sa + (uint32_t)(iy * kClaimPitch + ix) : scr_claim;
    vx[u] = __fmul_rn(-fx[u], dd[u]);
    vy[u] = __fmul_rn(-fy[u], dd[u]);
    dv[u] = dd[u];
  }
  int rounds = 0;
#pragma unroll 1
  for (;;) {
    claim_round2(pend[0], pend[1], claim_a[0], claim_a[1], (uint32_t)lane, (uint32_t)(32 + lane), cell_a[0], cell_a[1],
                 vx[0], vy[0], dv[0], vx[1], vy[1], dv[1], scr_cell, scr_claim);
    if (!__any_sync(0xffffffffu, (pend[0] | pend[1]) != 0)) break;
    // every round retires at least one source per contested cell: at most U * 32 rounds.  The guard turns a logic
    // error into a redo by the general path instead of a hung GPU.
    if (++rounds > U * 32 + 2) { vmax = __int_as_float(0x7f800000); break; }
  }
}

// A lane's share of a 16 x 16 source block: column pair 2j, 2j+1 (j = lane & 7) of the four rows 4g .. 4g+3
// (g = lane >> 3), held in the order k -> row 4g + ((k + rot) & 3), rot = 1 for the lanes j >= 4.  One load
// instruction covers 16 columns of four rows 4 apart (j < 4 and j >= 4 on neighbouring rows): 128-byte row segments.
// The rotation makes a claim round (below) bank-conflict free: the eight lanes of a quarter warp work on columns 2
// apart, the upper four one row below / above the lower four -> eight different 16-byte bank groups (129 cells a row).
struct BlockData {
  float4 f[4];      // flow of the pair: (fx, fy) of column 2j, (fx, fy) of column 2j+1
  float2 d[4];      // inverse depth of the pair
};

// The block loads are asm volatile so that they stay where they are written: AFTER touch_block() of the block about
// to be processed.  ncu on the first version (plain __ldg prefetch at the top of a phase): in two of the four phases
// ptxas had put the loads of both register buffers on the same scoreboard, so the first use of the block loaded a
// phase ago also waited for the loads issued a few instructions earlier -- ~1.8k cycles per block, every time.
__device__ __forceinline__ float4 ldg_nc_f4_v(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ float2 ldg_nc_f2_v(const float2* p) {
  float2 r;
  asm volatile("ld.global.nc.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  return r;
}

__device__ __forceinline__ void load_block(BlockData& s, const float2* __restrict__ flow, const float* __restrict__ depth,
                                           int h, int w, int bx0, int by0, int lane) {
  const int x = bx0 + 2 * (lane & 7), y0 = by0 + 4 * (lane >> 3), rot = (lane >> 2) & 1;
  if (bx0 >= 0 && by0 >= 0 && bx0 + kBS <= w && by0 + kBS <= h) {     // warp-uniform: the whole block is inside
    const int o0 = (y0 + rot) * w + x;
    const int o3 = o0 + (3 - 4 * rot) * w;
    const int off[4] = {o0, o0 + w, o0 + 2 * w, o3};
#pragma unroll
    for (int k = 0; k < 4; ++k) s.f[k] = ldg_nc_f4_v(reinterpret_cast<const float4*>(flow + off[k]));
#pragma unroll
    for (int k = 0; k < 4; ++k) s.d[k] = depth ? ldg_nc_f2_v(reinterpret_cast<const float2*>(depth + off[k])) : make_float2(1.0f, 1.0f);
    return;
  }
  const bool okx = (unsigned)x < (unsigned)w;       // w and x are even: the pair is inside or outside together
  const float qnan = __int_as_float(0x7fc00000);    // "no source": fails the range test, ignored by the bound check
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int y = y0 + ((k + rot) & 3);
    s.f[k] = make_float4(qnan, qnan, qnan, qnan);
    s.d[k] = make_float2(1.0f, 1.0f);
    if (okx && (unsigned)y < (unsigned)h) {
      const int off = y * w + x;
      s.f[k] = ldg_nc_f4_v(reinterpret_cast<const float4*>(flow + off));
      if (depth) s.d[k] = ldg_nc_f2_v(reinterpret_cast<const float2*>(depth + off));
    }
  }
}

// First use of every register of a block, as asm volatile (ordered before the next block's loads): the bound check
// (vmax = largest |flow component| seen; max ignores the NaN of "no source") and a running minimum of the inverse
// depths, whose only purpose is to read them here (its use at the end of the kernel can never change a result).
__device__ __forceinline__ void touch_block(const BlockData& s, float& vmax, float& dmin) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    asm volatile(
        "{\n .reg .f32 t0, t1;\n"
        " abs.f32 t0, %2;\n abs.f32 t1, %3;\n max.f32 t0, t0, t1;\n max.f32 %0, %0, t0;\n"
        " abs.f32 t0, %4;\n abs.f32 t1, %5;\n max.f32 t0, t0, t1;\n max.f32 %0, %0, t0;\n"
        " min.f32 t0, %6, %7;\n min.f32 %1, %1, t0;\n}"
        : "+f"(vmax), "+f"(dmin)
        : "f"(s.f[k].x), "f"(s.f[k].y), "f"(s.f[k].z), "f"(s.f[k].w), "f"(s.d[k].x), "f"(s.d[k].y));
  }
}

// Four claim rounds of 2 x 32 sources: (column parity p, k parity kb).  The 64 sources of a round are 2 apart in x
// and (within a lane group) in y: a smooth field (|gradient| < 0.5 px/px) practically never collides inside a round.
__device__ __forceinline__ void add_block(const BlockData& s, int bx0, int by0, uint32_t cells_sa, uint32_t claim_sa,
                                          const TileRect& R, int lane, float& vmax) {
  const float rotf = (float)((lane >> 2) & 1);
  const float xf0 = (float)(bx0 + 2 * (lane & 7));
  const float yr = (float)(by0 + 4 * (lane >> 3)) + rotf;              // row of k = 0
  const float yk[4] = {yr, yr + 1.0f, yr + 2.0f, fmaf(-4.0f, rotf, yr + 3.0f)};
#pragma unroll
  for (int p = 0; p < 2; ++p) {
#pragma unroll
    for (int kb = 0; kb < 2; ++kb) {
      float fx[2], fy[2], dd[2], xs[2], ys[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int k = kb + 2 * u;
        fx[u] = p ? s.f[k].z : s.f[k].x;
        fy[u] = p ? s.f[k].w : s.f[k].y;
        dd[u] = p ? s.d[k].y : s.d[k].x;
        xs[u] = xf0 + (float)p;
        ys[u] = yk[k];
      }
      add_sources<2, false>(fx, fy, dd, xs, ys, cells_sa, claim_sa, R, lane, vmax);
    }
  }
}

struct TilePos {
  int tb, tx0, ty0;
};
__device__ __forceinline__ TilePos tile_pos(int tile, int tiles_x, int tiles_xy) {
  TilePos t;
  t.tb = tile / tiles_xy;
  const int tr = tile - t.tb * tiles_xy;
  const int ty = tr / tiles_x;
  t.tx0 = (tr - ty * tiles_x) * kTW;
  t.ty0 = ty * kTH;
  return t;
}

template <bool WSUM>
__global__ void __launch_bounds__(kTileThreads, 1)
projection_tiled_kernel(const ProjArgs a) {
  extern __shared__ float4 s_cells[];
  uint32_t* s_colm = reinterpret_cast<uint32_t*>(s_cells + kNC + 32);          // [kColWords][kTW]
  const uint32_t cells_sa = (uint32_t)__cvta_generic_to_shared(s_cells);
  const uint32_t claim_sa = (uint32_t)__cvta_generic_to_shared(s_colm + kColWords * kTW);    // one claim byte per cell,
                                                                                             // kClaimPitch a row
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = a.h, w = a.w;
  const int tiles_x = ceil_div(w, kTW), tiles_xy = tiles_x * ceil_div(h, kTH);
  const int n_tiles = tiles_xy * a.B;
  const int P = h * w;                            // <= 2^30
  const float xmax = (float)(w - 1), ymax = (float)(h - 1);
  const int rw_x = ceil_div(w, 32);
  const int rw = h * rw_x, cw = ceil_div(h, 32) * w;
  const int n_halves = 2 * ceil_div(h, 32);       // 16-row halves of the column bitmap words
  const float2* flow_all = reinterpret_cast<const float2*>(a.flow);
  // super-block of this warp: block (2*sc + cx, 2*sr + cy) in colour phase (cx, cy)
  const int sc = warp % (kNBX / 2), sr = warp / (kNBX / 2);
  float vmax = 0.0f;                              // largest |flow component| this thread has looked at
  float dmin = __int_as_float(0x7f800000);        // see touch_block

  // the block of (tile, colour): origin and image
  auto block_org = [&](const TilePos& t, int c, int& bx0, int& by0) {
    bx0 = t.tx0 + kSX0 + kBS * (2 * sc + (c & 1));
    by0 = t.ty0 + kSY0 + kBS * (2 * sr + (c >> 1));
  };
  auto prefetch = [&](BlockData& s, int tile, int c) {
    if (tile >= n_tiles) return;
    const TilePos t = tile_pos(tile, tiles_x, tiles_xy);
    int bx0, by0;
    block_org(t, c, bx0, by0);
    load_block(s, flow_all + (int64_t)t.tb * P, a.inv_depth ? a.inv_depth + (int64_t)t.tb * P : nullptr, h, w, bx0, by0, lane);
  };

  for (int i = threadIdx.x; i < kColWords * kTW; i += kTileThreads) s_colm[i] = 0;
  for (int i = threadIdx.x; i < kNC; i += kTileThreads) s_cells[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  BlockData bufA, bufB;                           // the next block's loads fly under the current block's arithmetic
  if (warp < kAccWarps) prefetch(bufA, blockIdx.x, 0);

  // the extra source row of a tile (warp kAccWarps only): loaded one tile ahead like the blocks, added in phase 0
  float2 ex_f[kExtraChunks];
  float ex_d[kExtraChunks];
  auto load_extra = [&](int tile) {
    if (tile >= n_tiles) return;
    const TilePos t = tile_pos(tile, tiles_x, tiles_xy);
    const int ye = t.ty0 + kTH - 1 + kBD;
    if (ye >= h) return;
    const float2* flow = flow_all + (int64_t)t.tb * P;
#pragma unroll
    for (int ch = 0; ch < kExtraChunks; ++ch) {
      const int x = t.tx0 + kSX0 + 32 * ch + lane;
      ex_f[ch] = make_float2(__int_as_float(0x7fc00000), __int_as_float(0x7fc00000));
      ex_d[ch] = 1.0f;
      if ((unsigned)x < (unsigned)w) {
        ex_f[ch] = __ldg(flow + ye * w + x);
        if (a.inv_depth) ex_d[ch] = __ldg(a.inv_depth + (int64_t)t.tb * P + ye * w + x);
      }
    }
  };
  if (warp == kAccWarps) load_extra(blockIdx.x);

  int prev_tile = -1;
  auto flush_colm = [&](int tile) {               // column bitmap of a finished tile: 16-bit halves; re-zeroed
    const TilePos t = tile_pos(tile, tiles_x, tiles_xy);
    uint16_t* cm = reinterpret_cast<uint16_t*>(a.colmask + (int64_t)t.tb * cw);
    for (int i = threadIdx.x; i < kColWords * kTW; i += kTileThreads) {      // one staged word per thread
      const int wq = i / kTW, col = i - wq * kTW;
      const uint32_t word = s_colm[i];
      s_colm[i] = 0;
      const int x = t.tx0 + col;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int q = 2 * wq + e - ((t.ty0 & 31) >> 4);      // 16-row half of the tile held by this half word
        const int hy = t.ty0 / 16 + q;
        // the last tile row also writes the (empty) halves between the image's last row and the end of its bitmap word
        if (q >= 0 && (q < kTH / 16 || t.ty0 + kTH >= h) && x < w && hy < n_halves)
          cm[((hy >> 1) * w + x) * 2 + (hy & 1)] = (uint16_t)(word >> (16 * e));
      }
    }
  };

  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const TilePos t = tile_pos(tile, tiles_x, tiles_xy);
    const int tx0 = t.tx0, ty0 = t.ty0;
    if (prev_tile >= 0) flush_colm(prev_tile);
    prev_tile = tile;
    const int ye = ty0 + kTH - 1 + kBD;          // the extra source row (warp kAccWarps), loaded a tile ahead
    // the cells: the output pass of the previous tile cleared what only one warp reads; the rest -- the rows / columns
    // on the seams between the output warps and the halo row / column -- is cleared here
    for (int i = threadIdx.x; i < kSeamCells; i += kTileThreads) {
      int row, col;
      if (i < kSeamRows * kCW) {
        row = (i / kCW) * kOutRows;
        col = i % kCW;
      } else {
        const int j = i - kSeamRows * kCW;
        row = j / (kTW / 32 + 1);
        col = (j % (kTW / 32 + 1)) * 32;
      }
      s_cells[row * kCW + col] = make_float4(0.f, 0.f, 0.f, 0.f);
    }

    TileRect R;
    {
      // int(x2) in [lo, hi) <=> lo <= x2 < hi for x2 >= 0; `x2 < hi` is `x2 <= pred(hi)`, and at the image edge the
      // bound is Appendix B's x2 <= w-1
      const int gcx_hi = tx0 + kTW, gcy_hi = ty0 + kTH;
      R.xa = (float)max(tx0 - 1, 0);
      R.xb = gcx_hi <= w - 1 ? nextafterf((float)gcx_hi, 0.0f) : xmax;
      R.ya = (float)max(ty0 - 1, 0);
      R.yb = gcy_hi <= h - 1 ? nextafterf((float)gcy_hi, 0.0f) : ymax;
      R.cx0f = (float)(tx0 - 1);
      R.cy0f = (float)(ty0 - 1);
    }
    __syncthreads();

    // ---- accumulate: 4 colour phases
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      if (warp < kAccWarps) {
        BlockData& cur = (c & 1) ? bufB : bufA;
        BlockData& nxt = (c & 1) ? bufA : bufB;
        touch_block(cur, vmax, dmin);             // waits for the loads of a phase ago -- before the next ones go out
        if (c < 3) prefetch(nxt, tile, c + 1); else prefetch(nxt, tile + gridDim.x, 0);
        int bx0, by0;
        block_org(t, c, bx0, by0);
        if (bx0 < w && by0 < h && bx0 + kBS > 0 && by0 + kBS > 0)       // warp-uniform: the block touches the image
          add_block(cur, bx0, by0, cells_sa, claim_sa, R, lane, vmax);
      } else if (c == 0 && warp == kAccWarps && ye < h) {
        // the extra source row; no block active in phases 0 / 1 reaches the cell row it can hit
#pragma unroll
        for (int ch = 0; ch < kExtraChunks; ++ch) {
          float fx[1] = {ex_f[ch].x}, fy[1] = {ex_f[ch].y}, dd[1] = {ex_d[ch]};
          float xs[1] = {(float)(tx0 + kSX0 + 32 * ch + lane)}, ys[1] = {(float)ye};
          add_sources<1, true>(fx, fy, dd, xs, ys, cells_sa, claim_sa, R, lane, vmax);
        }
      }
      if (c == 0 && warp == kAccWarps) load_extra(tile + gridDim.x);
      __syncthreads();
    }

    // ---- output: warp = (32-column chunk, kOutRows target rows), lane = column; local cell of target (r, c) = (r+1, c+1)
    {
      const int chunk = warp & 3, r0 = (warp >> 2) * kOutRows;
      if (tx0 + 32 * chunk < w && ty0 + r0 < h) {
        const int x = tx0 + 32 * chunk + lane;
        const bool in_x = x < w;
        const float mx = (x == w - 1) ? 2.0f : 1.0f;
        float4* col = s_cells + r0 * kCW + 32 * chunk + lane + 1;           // cell row above the first target
        // horizontal pair sums h(r) = cell(r, x) * mx + cell(r, x-1); target = h(own row) * my + h(row above).  The
        // clamped duplicate targets of Appendix B ("hit twice") are the multiplicities mx, my of the last column / row.
        // Both cells come from shared memory (a second 16-byte load is cheaper than four shuffles and their moves).
        float4 hp;
        {
          const float4 c1 = col[0], c0 = col[-1];
          hp = make_float4(fmaf(c1.x, mx, c0.x), fmaf(c1.y, mx, c0.y), fmaf(c1.z, mx, c0.z), fmaf(c1.w, mx, c0.w));
        }
        uint32_t colbits = 0;
        uint32_t holerows = 0;                      // warp-uniform: rows of this chunk whose word has a hole
        const uint32_t inx_mask = __ballot_sync(0xffffffffu, in_x);
        const int rows = min(kOutRows, h - (ty0 + r0));
        const int64_t p0 = (int64_t)t.tb * P + (ty0 + r0) * w + x;
        float2* pp = reinterpret_cast<float2*>(a.proj) + p0;
        float* pw = WSUM ? a.wsum + p0 : nullptr;
        int32_t* pc = a.count + p0;
        uint8_t* ph = a.hole + p0;
        uint32_t* pr = a.rowmask + (int64_t)t.tb * rw + (ty0 + r0) * rw_x + ((tx0 + 32 * chunk) >> 5);
        const int r_last = h - 1 - (ty0 + r0);      // the image's last row, relative to this warp's first
        for (int r = 0; r < rows; ++r) {
          col += kCW;
          const float4 c1 = col[0], c0 = col[-1];
          // cleared for the next tile right here, except what another warp reads too (lane 31's own column is the next
          // chunk's left neighbour, the last row the next row group's row above): those cells wait for the barrier
          // (__syncwarp: the neighbouring lane's load of this cell as ITS left neighbour must come first)
          __syncwarp();
          if (lane < 31 && r < kOutRows - 1) col[0] = make_float4(0.f, 0.f, 0.f, 0.f);
          const float4 hc = make_float4(fmaf(c1.x, mx, c0.x), fmaf(c1.y, mx, c0.y), fmaf(c1.z, mx, c0.z), fmaf(c1.w, mx, c0.w));
          const float my = (r == r_last) ? 2.0f : 1.0f;
          const float4 tg = make_float4(fmaf(hc.x, my, hp.x), fmaf(hc.y, my, hp.y), fmaf(hc.z, my, hp.z), fmaf(hc.w, my, hp.w));
          hp = hc;
          float2 o;
          const bool is_hole = normalise_target_fast(tg, o);
          if (in_x) {
            *pp = o;
            if (WSUM) *pw = is_hole ? 0.0f : tg.z;
            *pc = (int32_t)tg.w;
            *ph = is_hole ? 1 : 0;
          }
          const uint32_t m = __ballot_sync(0xffffffffu, in_x && !is_hole);
          if (lane == 0) *pr = m;
          colbits |= (uint32_t)(in_x && !is_hole) << r;
          holerows |= (uint32_t)((inx_mask & ~m) != 0) << r;
          pp += w;
          if (WSUM) pw += w;
          pc += w;
          ph += w;
          pr += rw_x;
        }
        // this lane's column bits -> the staged column words (tile rows start at bit ty0 % 32 of the first word)
        const int pos = (ty0 & 31) + r0;
        const uint64_t bits = (uint64_t)colbits << (pos & 31);
        uint32_t* cmw = s_colm + (pos >> 5) * kTW + 32 * chunk + lane;
        if ((uint32_t)bits) atomicOr(cmw, (uint32_t)bits);
        if ((uint32_t)(bits >> 32)) atomicOr(cmw + kTW, (uint32_t)(bits >> 32));
        // the words with holes go on the list the fill kernel walks (one atomic per warp and tile)
        const int nh = __popc(holerows);
        if (nh > 0) {
          int base = 0;
          if (lane == 0) base = atomicAdd(a.flags + 1 + a.B, nh);
          base = __shfl_sync(0xffffffffu, base, 0);
          if (lane < nh) {
            const int r = __fns(holerows, 0, lane + 1);
            a.holelist[base + lane] = (uint32_t)(t.tb * rw + (ty0 + r0 + r) * rw_x + ((tx0 + 32 * chunk) >> 5));
          }
        }
      }
    }
    __syncthreads();
  }
  if (prev_tile >= 0) flush_colm(prev_tile);
  // a source beyond the bound: the colour phases may have raced and the scan may have missed cells it reaches -> the
  // whole batch is redone by the general path
  // (dmin: a value no sum of the comparison can produce keeps the reads of touch_block alive; if an inverse depth
  // ever were that denormal the batch would merely take the general path)
  if (__any_sync(0xffffffffu, vmax > (float)kBD || dmin == -1.0e-42f) && lane == 0) *reinterpret_cast<volatile int*>(a.flags) = 1;
}

// fill of the bounded path: the listed row words of all images in one launch; nothing at all when the promise was
// broken (the general path redoes the batch, its own fill included).  (The first version walked every row word of every
// image with holes: 64 us for eight 1080p images whose only holes sit at the image borders.)
__global__ void __launch_bounds__(kThreads)
projection_fill_kernel(const ProjArgs a) {
  if (*reinterpret_cast<volatile int*>(a.flags) != 0) return;
  const int lane = threadIdx.x & 31;
  const int nw = (gridDim.x * kThreads) >> 5;
  const int warp0 = (blockIdx.x * kThreads + threadIdx.x) >> 5;
  const int64_t P = (int64_t)a.h * a.w;
  const int rw = (int)rowmask_words(a.h, a.w);
  const int64_t cw = colmask_words(a.h, a.w);
  const int n = *reinterpret_cast<volatile int*>(a.flags + 1 + a.B);
  for (int i = warp0; i < n; i += nw) {
    const uint32_t gw = __ldg(a.holelist + i);
    const int b = (int)(gw / (uint32_t)rw), wd = (int)(gw - (uint32_t)b * (uint32_t)rw);
    fill_word<false>(a.rowmask + (int64_t)b * rw, a.colmask + b * cw, a.proj + b * P * 2, a.h, a.w, wd, lane);
  }
}

struct ProjWs {
  size_t acc_bytes, flags_off, row_off, col_off, list_off, total;
};
inline size_t up256(size_t v) { return (v + 255) / 256 * 256; }
inline ProjWs proj_ws(int B, int h, int w) {
  ProjWs s;
  s.acc_bytes = (size_t)h * w * sizeof(float4);
  s.flags_off = 3 * s.acc_bytes;
  s.row_off = s.flags_off + up256((size_t)(B + 2) * 4);
  s.col_off = s.row_off + up256((size_t)B * ceil_div(w, 32) * h * 4);
  s.list_off = s.col_off + up256((size_t)B * ceil_div(h, 32) * w * 4);
  s.total = s.list_off + up256((size_t)B * ceil_div(w, 32) * h * 4);
  return s;
}

// co-resident CTAs of the cooperative kernel on the current device
int pipeline_grid() {
  static int per_sm[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
  int sms = 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = kNumSMs;
  int occ = dev < 64 ? per_sm[dev] : 0;
  if (occ == 0) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, projection_pipeline_kernel, kThreads, 0) != cudaSuccess || occ < 1)
      occ = 1;
    if (dev < 64) per_sm[dev] = occ;
  }
  return sms * occ;
}

int launch_pipeline(const ProjArgs& a, cudaStream_t st) {
  ProjArgs args = a;
  void* kargs[] = {&args};
  int grid = pipeline_grid();
  // no more CTAs than there are warp tasks in the widest role (small images)
  const int64_t tasks = (int64_t)ceil_div(a.w, 32) * a.h;
  const int64_t want = ceil_div64(tasks, kThreads / 32);
  if (want < grid) grid = (int)(want < 1 ? 1 : want);
  cudaError_t e = cudaLaunchCooperativeKernel(reinterpret_cast<void*>(projection_pipeline_kernel), dim3(grid), dim3(kThreads),
                                              kargs, 0, st);
  if (e != cudaSuccess) return cuda_status(e);
  return after_launch();
}

// General path: per image memset -> splat -> normalise -> fill on the caller's stream, one L2-resident cell array.
// Measured alternatives on B200 (1080p, batch 8, us per image, smooth +-8 / i.i.d. +-64 / occlusion; profiles/
// time_ops_r02*.log): this sequence 45 / 59 / 45; images on 2 internal streams with 2 cell arrays 50 / 88 / 49; on 3
// streams 52 / 133 / 51 -- more than one 33 MB cell array in flight falls out of L2 under the streaming traffic and the
// scattered reductions go to DRAM; the whole batch pipelined inside one cooperative kernel (projection_pipeline_kernel
// above, kept as the fallback of the bounded path) 69 / 255 / 103 -- every role then runs at the merged kernel's 24
// warps per SM.
int run_general(const ProjArgs& a, cudaStream_t st) {
  const int h = a.h, w = a.w;
  const int64_t P = (int64_t)h * w;
  const int64_t rw = (int64_t)h * ceil_div(w, 32), cw = (int64_t)ceil_div(h, 32) * w;
  cudaError_t e = cudaMemsetAsync(a.flags + 1, 0, (size_t)a.B * 4, st);
  if (e != cudaSuccess) return cuda_status(e);
  const int n_tasks = ceil_div(w, 32) * ceil_div(h, kRows);
  const int splat_blocks = ceil_div(n_tasks, kThreads / 32);
  const int norm_blocks = ceil_div(ceil_div(w, 32) * (32 / kStrip) * ceil_div(h, 32), kThreads / 32);
  const int fill_blocks = min(ceil_div(h * ceil_div(w, 32), kThreads / 32), kNumSMs * 16);   // warps walk the hole list
  if ((e = cudaMemsetAsync(a.acc, 0, (size_t)P * sizeof(float4), st)) != cudaSuccess) return cuda_status(e);
  for (int b = 0; b < a.B; ++b) {
    int rc = launch_chained(stage_splat_kernel, splat_blocks, kThreads, st, a.flow + b * P * 2,
                            a.inv_depth ? a.inv_depth + b * P : nullptr, a.acc, h, w);
    if (rc) return rc;
    rc = launch_chained(stage_normalise_kernel, norm_blocks, kThreads, st, (const float4*)a.acc, a.proj + b * P * 2,
                        a.wsum ? a.wsum + b * P : nullptr, a.count + b * P, a.hole + b * P, a.rowmask + b * rw,
                        a.colmask + b * cw, a.flags + 1 + b, a.holelist + b * rw, h, w);
    if (rc) return rc;
    rc = launch_chained(stage_fill_kernel, fill_blocks, kThreads, st, (const uint32_t*)(a.rowmask + b * rw),
                        (const uint32_t*)(a.colmask + b * cw), (const int*)(a.flags + 1 + b),
                        (const uint32_t*)(a.holelist + b * rw), a.proj + b * P * 2, b + 1 < a.B ? a.acc : (float4*)nullptr, h, w);
    if (rc) return rc;
  }
  return VSR_OK;
}

}  // namespace

int launch_projection_fill(const uint32_t* rowmask, const uint32_t* colmask, const int* n_holewords,
                           const uint32_t* holelist, float* proj, int h, int w, cudaStream_t st) {
  const int fill_blocks = min(ceil_div(h * ceil_div(w, 32), kThreads / 32), kNumSMs * 16);
  stage_fill_kernel<<<fill_blocks, kThreads, 0, st>>>(rowmask, colmask, n_holewords, holelist, proj, nullptr, h, w);
  return after_launch();
}

}  // namespace vsr

using namespace vsr;

extern "C" size_t vsr_flow_projection_workspace_bytes(int B, int h, int w) {
  if (B <= 0 || h <= 0 || w <= 0) return 0;
  return proj_ws(B, h, w).total;
}

extern "C" int vsr_flow_projection_forward_bounded(const float* flow, const float* inv_depth, float* proj, float* wsum,
                                                   int32_t* count, uint8_t* hole, void* workspace, size_t workspace_bytes,
                                                   int B, int h, int w, float max_disp, vsr_stream_t stream) {
  if (!flow || !proj || !count || !hole || !workspace || B <= 0 || h <= 0 || w <= 0) return VSR_ERR_INVALID_ARG;
  if ((int64_t)h * w > (int64_t)1 << 30) return VSR_ERR_UNSUPPORTED;
  if (workspace_bytes < vsr_flow_projection_workspace_bytes(B, h, w)) return VSR_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(workspace) % 16 || reinterpret_cast<uintptr_t>(flow) % 8 ||
      reinterpret_cast<uintptr_t>(proj) % 8)
    return VSR_ERR_INVALID_ARG;
  cudaStream_t st = as_stream(stream);
  const ProjWs ws = proj_ws(B, h, w);
  uint8_t* base = reinterpret_cast<uint8_t*>(workspace);
  ProjArgs a;
  a.flow = flow;
  a.inv_depth = inv_depth;
  a.proj = proj;
  a.wsum = wsum;
  a.count = count;
  a.hole = hole;
  a.acc = reinterpret_cast<float4*>(base);
  a.flags = reinterpret_cast<int*>(base + ws.flags_off);
  a.rowmask = reinterpret_cast<uint32_t*>(base + ws.row_off);
  a.colmask = reinterpret_cast<uint32_t*>(base + ws.col_off);
  a.holelist = reinterpret_cast<uint32_t*>(base + ws.list_off);
  a.B = B;
  a.h = h;
  a.w = w;
  a.gate = 0;
  const bool bounded = max_disp >= 0.0f && max_disp <= (float)kMaxBound && w % 2 == 0 &&
                       reinterpret_cast<uintptr_t>(flow) % 16 == 0 && reinterpret_cast<uintptr_t>(inv_depth) % 8 == 0 &&
                       (int64_t)B * h * ceil_div(w, 32) < ((int64_t)1 << 31);   // NaN / negative / large, or
                                                                                       // unaligned pixel pairs (the tile path
                                                                                       // loads two pixels at a time): general path
  if (!bounded) return run_general(a, st);
  {
    // one tile per CTA and pass: between one and 1.75 waves of tiles (a single 1080p image: 210 tiles on 148 SMs) the
    // second, mostly empty pass costs more than the general path takes for the whole image (51 against 41 us)
    const int n_tiles = ceil_div(w, kTW) * ceil_div(h, kTH) * B;
    if (n_tiles > kNumSMs && n_tiles < kNumSMs * 7 / 4) return run_general(a, st);
  }

  static PerDeviceOnce once;
  int dev;
  if (once.needed(&dev)) {
    cudaError_t e = cudaFuncSetAttribute(projection_tiled_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTileSmem);
    if (e != cudaSuccess) return cuda_status(e);
    e = cudaFuncSetAttribute(projection_tiled_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTileSmem);
    if (e != cudaSuccess) return cuda_status(e);
    once.mark(dev);
  }
  cudaError_t e = cudaMemsetAsync(a.flags, 0, (size_t)(B + 2) * 4, st);
  if (e != cudaSuccess) return cuda_status(e);
  const int n_tiles = ceil_div(w, kTW) * ceil_div(h, kTH) * B;
  if (wsum)
    projection_tiled_kernel<true><<<n_tiles < kNumSMs ? n_tiles : kNumSMs, kTileThreads, kTileSmem, st>>>(a);
  else
    projection_tiled_kernel<false><<<n_tiles < kNumSMs ? n_tiles : kNumSMs, kTileThreads, kTileSmem, st>>>(a);
  int rc = after_launch();
  if (rc) return rc;
  const int64_t fill_warps = (int64_t)h * ceil_div(w, 32);
  int64_t fill_blocks = ceil_div64(fill_warps, kThreads / 32);
  if (fill_blocks > kNumSMs * 16) fill_blocks = kNumSMs * 16;
  projection_fill_kernel<<<(int)fill_blocks, kThreads, 0, st>>>(a);
  rc = after_launch();
  if (rc) return rc;
  a.gate = 1;   // the whole batch again through the general path, only if a source broke the promise
  return launch_pipeline(a, st);
}

extern "C" int vsr_flow_projection_forward(const float* flow, const float* inv_depth, float* proj, float* wsum,
                                           int32_t* count, uint8_t* hole, void* workspace, size_t workspace_bytes,
                                           int B, int h, int w, vsr_stream_t stream) {
  return vsr_flow_projection_forward_bounded(flow, inv_depth, proj, wsum, count, hole, workspace, workspace_bytes, B, h,
                                             w, -1.0f, stream);
}
