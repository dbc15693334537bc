// deterministic.cu -- run-to-run deterministic flow projection (a1 / a2) and Resample2d input gradient, bit-identical
// to the CPU restatement (oracle/oracle.c: or_flow_projection, or_resample2d_backward).
//
// The default kernels of both ops scatter with fp32 atomics (projection.cu's general path, warp.cu's
// resample2d_backward_input1_kernel), so the sums come out in arrival order.  Here each scatter becomes a gather that
// performs the oracle's additions in the oracle's order:
//   1. every source gets the key of its cell -- (int(y2), int(x2)) of its target for the projection (out-of-image and
//      NaN sources get the sentinel key h*w), the clamped top-left tap (b, yT, xL) for the resample gradient -- and the
//      sources per cell are counted (integer atomics: the counts do not depend on order);
//   2. a stable LSD radix sort of the source indices by key, 11 bits a pass (two passes cover a 1080p image).  Every
//      block ranks its tile of 4096 in a fixed order (warp after warp, lane after lane) and the (digit x block)
//      histograms are scanned digit-major, so each cell's list comes out in ascending source index: no per-cell sort,
//      and a cell that receives every source of the image needs no special case;
//   3. an exclusive scan of the per-cell counts gives each cell's range of the sorted list;
//   4. one thread per target merges the lists of the (up to) four cells whose sources can reach it, by source index,
//      and accumulates in that order -- in fp64 for the projection (the oracle's double sums of fp32 contributions),
//      in fp32 for the gradient.
// The projection then normalises with an IEEE divide, writes the occupancy bitmaps and the list of row words with
// holes, and reuses the general path's fill stage (its left, right, up, down fp32 sum and division by the number found
// are the oracle's).  The gradient w.r.t. the flow comes from warp.cu's kernel, which is already deterministic.
#include "common.cuh"

namespace vsr {
namespace {

constexpr int kSortThreads = 256;
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kRounds = 16;                              // 32-key rounds per warp
constexpr int kPerWarp = 32 * kRounds;                   // 512 keys: a warp's contiguous share of a tile
constexpr int kTile = kSortWarps * kPerWarp;             // 4096 keys per block
constexpr int kDigitBits = 11;
constexpr int kDigits = 1 << kDigitBits;
constexpr int kScanThreads = 1024;
constexpr int kScanItems = 8;
constexpr int kScanChunk = kScanThreads * kScanItems;
constexpr uint32_t kNone = 0xffffffffu;                  // "list exhausted": larger than every source index

// ---------------------------------------------------------------------------------------------
// Exclusive scan of n u32 (n up to 2^32 + 1 entries; the total must fit in u32).
// ---------------------------------------------------------------------------------------------
// Block-wide exclusive scan of one value per thread (kScanThreads threads); `total` receives the block's sum.
__device__ __forceinline__ uint32_t block_scan_excl(uint32_t v, uint32_t* s_warp, uint32_t& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += t;
  }
  if (lane == 31) s_warp[warp] = x;
  __syncthreads();
  if (warp == 0) {
    uint32_t y = s_warp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, y, o);
      if (lane >= o) y += t;
    }
    s_warp[lane] = y;
  }
  __syncthreads();
  const uint32_t before = warp ? s_warp[warp - 1] : 0u;
  total = s_warp[31];
  __syncthreads();   // s_warp is reused by the next call
  return before + x - v;
}

// One chunk of kScanChunk entries starting at `base`, offset by `carry`; returns the chunk's sum.  `in` may equal `out`.
__device__ __forceinline__ uint32_t scan_chunk(const uint32_t* in, uint32_t* out, int64_t n, int64_t base, uint32_t carry,
                                               uint32_t* s_warp) {
  uint32_t item[kScanItems];
  uint32_t sum = 0;
  const int64_t i0 = base + (int64_t)threadIdx.x * kScanItems;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    item[j] = i0 + j < n ? in[i0 + j] : 0u;
    sum += item[j];
  }
  uint32_t total;
  uint32_t run = carry + block_scan_excl(sum, s_warp, total);
  if (out) {
#pragma unroll
    for (int j = 0; j < kScanItems; ++j) {
      if (i0 + j < n) out[i0 + j] = run;
      run += item[j];
    }
  }
  return total;
}

// chunk sums -> part[chunk]
__global__ void __launch_bounds__(kScanThreads) det_scan_reduce_kernel(const uint32_t* in, int64_t n, uint32_t* part) {
  __shared__ uint32_t s_warp[32];
  const uint32_t t = scan_chunk(in, nullptr, n, (int64_t)blockIdx.x * kScanChunk, 0u, s_warp);
  if (threadIdx.x == 0) part[blockIdx.x] = t;
}

// chunk_off == nullptr: one block scans all n entries chunk after chunk (the chunk sums); otherwise block k scans
// chunk k starting from chunk_off[k]
__global__ void __launch_bounds__(kScanThreads) det_scan_kernel(const uint32_t* in, uint32_t* out, int64_t n,
                                                                const uint32_t* chunk_off) {
  __shared__ uint32_t s_warp[32];
  if (chunk_off) {
    scan_chunk(in, out, n, (int64_t)blockIdx.x * kScanChunk, chunk_off[blockIdx.x], s_warp);
    return;
  }
  uint32_t carry = 0;
  for (int64_t base = 0; base < n; base += kScanChunk) carry += scan_chunk(in, out, n, base, carry, s_warp);
}

inline int64_t scan_chunks(int64_t n) { return ceil_div64(n, kScanChunk); }

int exclusive_scan(const uint32_t* in, uint32_t* out, int64_t n, uint32_t* part, cudaStream_t st) {
  const int64_t nc = scan_chunks(n);
  det_scan_reduce_kernel<<<(unsigned)nc, kScanThreads, 0, st>>>(in, n, part);
  int rc = after_launch();
  if (rc) return rc;
  det_scan_kernel<<<1, kScanThreads, 0, st>>>(part, part, nc, nullptr);
  if ((rc = after_launch())) return rc;
  det_scan_kernel<<<(unsigned)nc, kScanThreads, 0, st>>>(in, out, n, part);
  return after_launch();
}

// ---------------------------------------------------------------------------------------------
// Stable LSD radix sort of (key, source index) pairs, kDigitBits per pass.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t digit_of(uint32_t key, int shift) { return (key >> shift) & (kDigits - 1); }

// hist[d * nblk + block] = number of keys of the block's tile with digit d
__global__ void __launch_bounds__(kSortThreads)
det_radix_hist_kernel(const uint32_t* __restrict__ keys, int64_t n, int shift, uint32_t* __restrict__ hist) {
  __shared__ uint32_t cnt[kDigits];
  for (int d = threadIdx.x; d < kDigits; d += kSortThreads) cnt[d] = 0;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * kTile;
  for (int i = threadIdx.x; i < kTile; i += kSortThreads)
    if (base + i < n) atomicAdd(&cnt[digit_of(__ldg(keys + base + i), shift)], 1u);
  __syncthreads();
  for (int d = threadIdx.x; d < kDigits; d += kSortThreads) hist[(int64_t)d * gridDim.x + blockIdx.x] = cnt[d];
}

// Scatter of one tile to its sorted positions.  off = the digit-major exclusive scan of hist: where the block's keys
// of digit d start.  Inside the block a key's rank is (keys of its digit in earlier warps) + (in earlier rounds of its
// warp) + (in lower lanes of its round): the tile order, so the pass is stable.  vals_in == nullptr: the values are
// the key indices (the first pass).
__global__ void __launch_bounds__(kSortThreads)
det_radix_scatter_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                         uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out, int64_t n, int shift,
                         const uint32_t* __restrict__ off) {
  __shared__ uint16_t s_wpos[kSortWarps][kDigits];   // per warp: its keys of digit d so far, then its start in the block
  __shared__ uint32_t s_boff[kDigits];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < kSortWarps * kDigits; i += kSortThreads) (&s_wpos[0][0])[i] = 0;
  for (int d = threadIdx.x; d < kDigits; d += kSortThreads) s_boff[d] = off[(int64_t)d * gridDim.x + blockIdx.x];
  __syncthreads();
  const int64_t i0 = (int64_t)blockIdx.x * kTile + warp * kPerWarp + lane;
  uint32_t key[kRounds];
#pragma unroll
  for (int r = 0; r < kRounds; ++r) {
    const int64_t i = i0 + 32 * r;
    key[r] = i < n ? __ldg(keys_in + i) : 0u;
  }
  // counts per warp and digit
#pragma unroll
  for (int r = 0; r < kRounds; ++r) {
    const bool valid = i0 + 32 * r < n;
    const uint32_t d = valid ? digit_of(key[r], shift) : (uint32_t)kDigits;
    const uint32_t peers = __match_any_sync(0xffffffffu, d);
    if (valid && lane == __ffs(peers) - 1) s_wpos[warp][d] += (uint16_t)__popc(peers);
    __syncwarp();
  }
  __syncthreads();
  // exclusive prefix over the warps, per digit (at most kTile: fits 16 bits)
  for (int d = threadIdx.x; d < kDigits; d += kSortThreads) {
    uint32_t run = 0;
#pragma unroll
    for (int wq = 0; wq < kSortWarps; ++wq) {
      const uint32_t c = s_wpos[wq][d];
      s_wpos[wq][d] = (uint16_t)run;
      run += c;
    }
  }
  __syncthreads();
  const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
  for (int r = 0; r < kRounds; ++r) {
    const int64_t i = i0 + 32 * r;
    const bool valid = i < n;
    const uint32_t d = valid ? digit_of(key[r], shift) : (uint32_t)kDigits;
    const uint32_t peers = __match_any_sync(0xffffffffu, d);
    uint32_t local = 0;
    if (valid) local = s_wpos[warp][d];
    __syncwarp();
    if (valid && lane == __ffs(peers) - 1) s_wpos[warp][d] = (uint16_t)(local + __popc(peers));
    __syncwarp();
    if (valid) {
      const uint32_t pos = s_boff[d] + local + __popc(peers & lt);
      keys_out[pos] = key[r];
      vals_out[pos] = vals_in ? __ldg(vals_in + i) : (uint32_t)i;
    }
  }
}

struct SortBufs {
  uint32_t* keys[2];    // keys[0]: the unsorted keys on entry
  uint32_t* vals[2];
  uint32_t* hist;       // kDigits * blocks
  uint32_t* part;       // chunk sums of the scans
};

inline int64_t sort_blocks(int64_t n) { return ceil_div64(n, kTile); }

// Sorts keys[0] (n keys <= max_key, with their indices as values); *sorted = the source indices in key order.
int radix_sort(const SortBufs& s, int64_t n, uint32_t max_key, cudaStream_t st, const uint32_t** sorted) {
  const int bits = max_key ? 32 - __builtin_clz(max_key) : 1;
  const int passes = ceil_div(bits, kDigitBits);
  const int64_t nblk = sort_blocks(n);
  for (int p = 0; p < passes; ++p) {
    const uint32_t* kin = s.keys[p & 1];
    const uint32_t* vin = p ? s.vals[(p + 1) & 1] : nullptr;
    det_radix_hist_kernel<<<(unsigned)nblk, kSortThreads, 0, st>>>(kin, n, p * kDigitBits, s.hist);
    int rc = after_launch();
    if (rc) return rc;
    if ((rc = exclusive_scan(s.hist, s.hist, (int64_t)kDigits * nblk, s.part, st))) return rc;
    det_radix_scatter_kernel<<<(unsigned)nblk, kSortThreads, 0, st>>>(kin, vin, s.keys[(p + 1) & 1], s.vals[p & 1], n,
                                                                       p * kDigitBits, s.hist);
    if ((rc = after_launch())) return rc;
  }
  *sorted = s.vals[(passes - 1) & 1];
  return VSR_OK;
}

// Workspace of one sort of n keys over ncells cells: 4 key / value arrays, the per-cell counts (ncells + 1), the
// histograms and the chunk sums; `extra` bytes follow for the caller.
struct SortWs {
  size_t keys[2], vals[2], start, hist, part, total;
};
inline size_t up256(size_t v) { return (v + 255) / 256 * 256; }
inline SortWs sort_ws(int64_t n, int64_t ncells) {
  SortWs s;
  const int64_t hist_n = (int64_t)kDigits * sort_blocks(n);
  const int64_t scan_n = hist_n > ncells + 1 ? hist_n : ncells + 1;
  size_t o = 0;
  for (int k = 0; k < 2; ++k) { s.keys[k] = o; o += up256((size_t)n * 4); }
  for (int k = 0; k < 2; ++k) { s.vals[k] = o; o += up256((size_t)n * 4); }
  s.start = o; o += up256((size_t)(ncells + 1) * 4);
  s.hist = o; o += up256((size_t)hist_n * 4);
  s.part = o; o += up256((size_t)scan_chunks(scan_n) * 4);
  s.total = o;
  return s;
}
inline SortBufs sort_bufs(const SortWs& s, uint8_t* base) {
  SortBufs b;
  for (int k = 0; k < 2; ++k) {
    b.keys[k] = reinterpret_cast<uint32_t*>(base + s.keys[k]);
    b.vals[k] = reinterpret_cast<uint32_t*>(base + s.vals[k]);
  }
  b.hist = reinterpret_cast<uint32_t*>(base + s.hist);
  b.part = reinterpret_cast<uint32_t*>(base + s.part);
  return b;
}

// ---------------------------------------------------------------------------------------------
// Flow projection
// ---------------------------------------------------------------------------------------------
// cell key of every source (Appendix B step 2; the comparison form also rejects NaN), sources per cell
__global__ void __launch_bounds__(kSortThreads)
det_proj_keys_kernel(const float2* __restrict__ flow, uint32_t* __restrict__ keys, uint32_t* __restrict__ cell_count,
                     int h, int w) {
  const int64_t P = (int64_t)h * w;
  const float xmax = (float)(w - 1), ymax = (float)(h - 1);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (int64_t)gridDim.x * blockDim.x) {
    const int y = (int)(i / w), x = (int)(i - (int64_t)y * w);
    const float2 f = __ldg(flow + i);
    const float x2 = __fadd_rn((float)x, f.x), y2 = __fadd_rn((float)y, f.y);
    uint32_t key = (uint32_t)P;
    if (x2 >= 0.0f && x2 <= xmax && y2 >= 0.0f && y2 <= ymax) {
      key = (uint32_t)((int)y2 * w + (int)x2);
      atomicAdd(cell_count + key, 1u);
    }
    keys[i] = key;
  }
}

// Lowest source index of the lists still open; k = its list.
__device__ __forceinline__ uint32_t merge_min(const uint32_t (&cur)[4], int& k) {
  uint32_t s = cur[0];
  k = 0;
#pragma unroll
  for (int j = 1; j < 4; ++j)
    if (cur[j] < s) {
      s = cur[j];
      k = j;
    }
  return s;
}
__device__ __forceinline__ void merge_advance(uint32_t (&cur)[4], uint32_t (&pos)[4], const uint32_t (&end)[4], int k,
                                              const uint32_t* __restrict__ src) {
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (j == k) {
      ++pos[j];
      cur[j] = pos[j] < end[j] ? __ldg(src + pos[j]) : kNone;
    }
}

// One thread per target; a warp = 32 columns of one row, a block = a 32 x 32 tile (the column bitmap words).  The
// target's sources sit in the cells (y-1|y, x-1|x); a source of cell (cy, cx) hits it mx * my times, mx = [cx == x] +
// [min(cx+1, w-1) == x] (the oracle's clamped duplicate at the last column / row).  Each source's (cx, cy, d) is added
// that many times in a row, in source order, in fp64.
constexpr int kGatherRowsPerWarp = 32 / kSortWarps;
__global__ void __launch_bounds__(kSortThreads)
det_proj_gather_kernel(const float2* __restrict__ flow, const float* __restrict__ inv_depth,
                       const uint32_t* __restrict__ src, const uint32_t* __restrict__ start, float2* __restrict__ proj,
                       float* __restrict__ wsum, int32_t* __restrict__ count, uint8_t* __restrict__ hole,
                       uint32_t* __restrict__ rowmask, uint32_t* __restrict__ colmask, int* __restrict__ n_holewords,
                       uint32_t* __restrict__ holelist, int h, int w) {
  __shared__ uint32_t s_col[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int x = blockIdx.x * 32 + lane;
  const int wpr = ceil_div(w, 32);
  if (threadIdx.x < 32) s_col[threadIdx.x] = 0;
  __syncthreads();
  const bool in_x = x < w;
  const uint32_t inx_mask = __ballot_sync(0xffffffffu, in_x);
  for (int r = 0; r < kGatherRowsPerWarp; ++r) {
    const int y = blockIdx.y * 32 + warp * kGatherRowsPerWarp + r;
    if (y >= h) break;                              // warp-uniform
    bool is_hole = true;
    if (in_x) {
      uint32_t pos[4], end[4], cur[4];
      int mult[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int cy = y - 1 + (k >> 1), cx = x - 1 + (k & 1);
        const int mx = (cx == x) + (min(cx + 1, w - 1) == x), my = (cy == y) + (min(cy + 1, h - 1) == y);
        mult[k] = mx * my;
        pos[k] = end[k] = 0;
        if (cx >= 0 && cy >= 0 && mult[k] > 0) {
          const int64_t c = (int64_t)cy * w + cx;
          pos[k] = __ldg(start + c);
          end[k] = __ldg(start + c + 1);
        }
        cur[k] = pos[k] < end[k] ? __ldg(src + pos[k]) : kNone;
      }
      double ax = 0.0, ay = 0.0, aw = 0.0;
      int cnt = 0;
      for (;;) {
        int k;
        const uint32_t s = merge_min(cur, k);
        if (s == kNone) break;
        const float2 f = __ldg(flow + s);
        const float d = inv_depth ? __ldg(inv_depth + s) : 1.0f;
        const double cx = (double)__fmul_rn(-f.x, d), cy = (double)__fmul_rn(-f.y, d), dd = (double)d;
        int m = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) m = j == k ? mult[j] : m;
        for (int t = 0; t < m; ++t) {
          ax = __dadd_rn(ax, cx);
          ay = __dadd_rn(ay, cy);
          aw = __dadd_rn(aw, dd);
        }
        cnt += m;
        merge_advance(cur, pos, end, k, src);
      }
      const float ws = __double2float_rn(aw);
      is_hole = !(cnt > 0 && ws > 0.0f);
      const int64_t p = (int64_t)y * w + x;
      proj[p] = is_hole ? make_float2(0.f, 0.f)
                        : make_float2(__fdiv_rn(__double2float_rn(ax), ws), __fdiv_rn(__double2float_rn(ay), ws));
      if (wsum) wsum[p] = is_hole ? 0.0f : ws;
      count[p] = cnt;
      hole[p] = is_hole ? 1 : 0;
    }
    const uint32_t m = __ballot_sync(0xffffffffu, in_x && !is_hole);
    if (lane == 0) {
      rowmask[y * wpr + blockIdx.x] = m;
      // the fill writes hole pixels only and reads non-hole pixels only: the list's order does not matter
      if (inx_mask & ~m) holelist[atomicAdd(n_holewords, 1)] = (uint32_t)(y * wpr + blockIdx.x);
    }
    if (in_x && !is_hole) atomicOr(&s_col[lane], 1u << (y & 31));
  }
  __syncthreads();
  if (threadIdx.x < 32 && in_x) colmask[blockIdx.y * w + x] = s_col[threadIdx.x];
}

// The per-image buffers after the sort's: row / column occupancy bitmaps, hole-word list and its length.
struct DetProjWs {
  SortWs sort;
  size_t row_off, col_off, list_off, nlist_off, total;
};
inline DetProjWs det_proj_ws(int h, int w) {
  DetProjWs s;
  const int64_t P = (int64_t)h * w;
  s.sort = sort_ws(P, P);
  s.row_off = s.sort.total;
  s.col_off = s.row_off + up256((size_t)h * ceil_div(w, 32) * 4);
  s.list_off = s.col_off + up256((size_t)ceil_div(h, 32) * w * 4);
  s.nlist_off = s.list_off + up256((size_t)h * ceil_div(w, 32) * 4);
  s.total = s.nlist_off + 256;
  return s;
}

// ---------------------------------------------------------------------------------------------
// Resample2d gradient w.r.t. input1 (kernel_size 1)
// ---------------------------------------------------------------------------------------------
// Taps and weights of source (b, y, x), computed exactly as resample2d_backward_input1_kernel does (warp.cu).
struct Taps {
  int xL, xR, yT, yB;
  float w[4];   // TL, TR, BL, BR
};
__device__ __forceinline__ Taps resample_taps(const float* __restrict__ flow, int64_t HW, int b, int y, int x, int H,
                                              int W) {
  const float* fl = flow + (int64_t)b * 2 * HW + (int64_t)y * W + x;
  const float dx = __ldg(fl), dy = __ldg(fl + HW);
  const float xf = __fadd_rn((float)x, dx), yf = __fadd_rn((float)y, dy);
  const float alpha = __fsub_rn(xf, (float)__float2int_rz(xf));     // int(), not floor (resample2d_kernel.cu:105-106)
  const float beta = __fsub_rn(yf, (float)__float2int_rz(yf));
  Taps t;
  t.xL = max(min((int)floorf(xf), W - 1), 0);
  t.xR = max(min((int)__fadd_rn(floorf(xf), 1.0f), W - 1), 0);
  t.yT = max(min((int)floorf(yf), H - 1), 0);
  t.yB = max(min((int)__fadd_rn(floorf(yf), 1.0f), H - 1), 0);
  const float ia = __fsub_rn(1.0f, alpha), ib = __fsub_rn(1.0f, beta);
  t.w[0] = __fmul_rn(ia, ib);
  t.w[1] = __fmul_rn(alpha, ib);
  t.w[2] = __fmul_rn(ia, beta);
  t.w[3] = __fmul_rn(alpha, beta);
  return t;
}

// key of every source: its clamped top-left tap (b, yT, xL); sources per cell
__global__ void __launch_bounds__(kSortThreads)
det_resample_keys_kernel(const float* __restrict__ flow, uint32_t* __restrict__ keys, uint32_t* __restrict__ cell_count,
                         int B, int H, int W, const PixDecode pd) {
  const int64_t HW = (int64_t)H * W, n = (int64_t)B * HW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int b, y, x;
    decode_pix((uint32_t)i, pd, b, y, x);
    const Taps t = resample_taps(flow, HW, b, y, x, H, W);
    const uint32_t key = (uint32_t)((int64_t)b * HW + (int64_t)t.yT * W + t.xL);
    atomicAdd(cell_count + key, 1u);
    keys[i] = key;
  }
}

// One thread per target (b, y, x).  xR is xL or xL + 1 and yB is yT or yT + 1 even after clamping, so the target's
// sources sit in the cells (b, y-1|y, x-1|x).  For kChanChunk channels at a time the thread walks the merged list and,
// for each source, adds w * g for each of its taps TL, TR, BL, BR that is the target, in that order, in fp32: the
// oracle's sequence.  Every element of grad_input1 is written.
constexpr int kChanChunk = 8;
__global__ void __launch_bounds__(kSortThreads)
det_resample_gather_kernel(const float* __restrict__ flow, const float* __restrict__ gout, const uint32_t* __restrict__ src,
                           const uint32_t* __restrict__ start, float* __restrict__ gin1, int B, int C, int H, int W,
                           const PixDecode pd) {
  const int64_t HW = (int64_t)H * W, n = (int64_t)B * HW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int b, y, x;
    decode_pix((uint32_t)i, pd, b, y, x);
    uint32_t pos0[4], end[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int cy = y - 1 + (k >> 1), cx = x - 1 + (k & 1);
      pos0[k] = end[k] = 0;
      if (cx >= 0 && cy >= 0) {
        const int64_t c = (int64_t)b * HW + (int64_t)cy * W + cx;
        pos0[k] = __ldg(start + c);
        end[k] = __ldg(start + c + 1);
      }
    }
    for (int c0 = 0; c0 < C; c0 += kChanChunk) {
      float acc[kChanChunk];
#pragma unroll
      for (int c = 0; c < kChanChunk; ++c) acc[c] = 0.0f;
      uint32_t pos[4], cur[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        pos[k] = pos0[k];
        cur[k] = pos[k] < end[k] ? __ldg(src + pos[k]) : kNone;
      }
      for (;;) {
        int k;
        const uint32_t s = merge_min(cur, k);
        if (s == kNone) break;
        int sb, sy, sx;
        decode_pix(s, pd, sb, sy, sx);
        const Taps t = resample_taps(flow, HW, sb, sy, sx, H, W);
        const bool hit[4] = {t.yT == y && t.xL == x, t.yT == y && t.xR == x, t.yB == y && t.xL == x,
                             t.yB == y && t.xR == x};
        const float* g = gout + ((int64_t)sb * C + c0) * HW + (int64_t)sy * W + sx;
#pragma unroll
        for (int c = 0; c < kChanChunk; ++c) {
          if (c0 + c < C) {
            const float gv = __ldg(g + (int64_t)c * HW);
#pragma unroll
            for (int q = 0; q < 4; ++q)
              if (hit[q]) acc[c] = __fadd_rn(acc[c], __fmul_rn(t.w[q], gv));
          }
        }
        merge_advance(cur, pos, end, k, src);
      }
      float* o = gin1 + ((int64_t)b * C + c0) * HW + (int64_t)y * W + x;
#pragma unroll
      for (int c = 0; c < kChanChunk; ++c)
        if (c0 + c < C) o[(int64_t)c * HW] = acc[c];
    }
  }
}

inline int grid_of(int64_t items) {
  const int64_t cap = (int64_t)kNumSMs * 8 * 4, blocks = ceil_div64(items, kSortThreads);
  return (int)(blocks < 1 ? 1 : blocks > cap ? cap : blocks);
}

}  // namespace
}  // namespace vsr

using namespace vsr;

extern "C" size_t vsr_flow_projection_deterministic_workspace_bytes(int B, int h, int w) {
  if (B <= 0 || h <= 0 || w <= 0) return 0;
  return det_proj_ws(h, w).total;   // one image at a time
}

extern "C" int vsr_flow_projection_forward_deterministic(const float* flow, const float* inv_depth, float* proj,
                                                         float* wsum, int32_t* count, uint8_t* hole, void* workspace,
                                                         size_t workspace_bytes, int B, int h, int w,
                                                         vsr_stream_t stream) {
  if (!flow || !proj || !count || !hole || !workspace || B <= 0 || h <= 0 || w <= 0) return VSR_ERR_INVALID_ARG;
  if ((int64_t)h * w > (int64_t)1 << 30) return VSR_ERR_UNSUPPORTED;
  if (workspace_bytes < vsr_flow_projection_deterministic_workspace_bytes(B, h, w)) return VSR_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(workspace) % 16 || reinterpret_cast<uintptr_t>(flow) % 8 ||
      reinterpret_cast<uintptr_t>(proj) % 8)
    return VSR_ERR_INVALID_ARG;
  cudaStream_t st = as_stream(stream);
  const DetProjWs ws = det_proj_ws(h, w);
  uint8_t* base = reinterpret_cast<uint8_t*>(workspace);
  const SortBufs sb = sort_bufs(ws.sort, base);
  uint32_t* start = reinterpret_cast<uint32_t*>(base + ws.sort.start);
  uint32_t* rowmask = reinterpret_cast<uint32_t*>(base + ws.row_off);
  uint32_t* colmask = reinterpret_cast<uint32_t*>(base + ws.col_off);
  uint32_t* holelist = reinterpret_cast<uint32_t*>(base + ws.list_off);
  int* n_holewords = reinterpret_cast<int*>(base + ws.nlist_off);
  const int64_t P = (int64_t)h * w;
  const dim3 gather_grid((unsigned)ceil_div(w, 32), (unsigned)ceil_div(h, 32));
  for (int b = 0; b < B; ++b) {
    const float2* fl = reinterpret_cast<const float2*>(flow) + b * P;
    const float* dp = inv_depth ? inv_depth + b * P : nullptr;
    cudaError_t e = cudaMemsetAsync(start, 0, (size_t)(P + 1) * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(n_holewords, 0, 4, st);
    if (e != cudaSuccess) return cuda_status(e);
    det_proj_keys_kernel<<<grid_of(P), kSortThreads, 0, st>>>(fl, sb.keys[0], start, h, w);
    int rc = after_launch();
    if (rc) return rc;
    const uint32_t* sorted;
    if ((rc = radix_sort(sb, P, (uint32_t)P, st, &sorted))) return rc;
    if ((rc = exclusive_scan(start, start, P + 1, sb.part, st))) return rc;
    det_proj_gather_kernel<<<gather_grid, kSortThreads, 0, st>>>(
        fl, dp, sorted, start, reinterpret_cast<float2*>(proj) + b * P, wsum ? wsum + b * P : nullptr, count + b * P,
        hole + b * P, rowmask, colmask, n_holewords, holelist, h, w);
    if ((rc = after_launch())) return rc;
    if ((rc = launch_projection_fill(rowmask, colmask, n_holewords, holelist, proj + b * P * 2, h, w, st))) return rc;
  }
  return VSR_OK;
}

extern "C" size_t vsr_resample2d_backward_deterministic_workspace_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  const int64_t n = (int64_t)B * H * W;
  return sort_ws(n, n).total;
}

extern "C" int vsr_resample2d_backward_deterministic(const float* input1, const float* flow, const float* grad_output,
                                                     float* grad_input1, float* grad_input2, int B, int C, int H, int W,
                                                     int kernel_size, int bilinear, void* workspace,
                                                     size_t workspace_bytes, vsr_stream_t stream) {
  (void)bilinear;  // ignored by the reference's backward as well
  if (!input1 || !flow || !grad_output || !grad_input1 || !grad_input2 || !workspace || B <= 0 || C <= 0 || H <= 0 ||
      W <= 0)
    return VSR_ERR_INVALID_ARG;
  if (kernel_size != 1) return VSR_ERR_UNSUPPORTED;
  if ((int64_t)B * H * W >= ((int64_t)1 << 32)) return VSR_ERR_UNSUPPORTED;
  if (workspace_bytes < vsr_resample2d_backward_deterministic_workspace_bytes(B, H, W)) return VSR_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(workspace) % 16) return VSR_ERR_INVALID_ARG;
  cudaStream_t st = as_stream(stream);
  const int64_t n = (int64_t)B * H * W;
  const SortWs ws = sort_ws(n, n);
  uint8_t* base = reinterpret_cast<uint8_t*>(workspace);
  const SortBufs sb = sort_bufs(ws, base);
  uint32_t* start = reinterpret_cast<uint32_t*>(base + ws.start);
  const PixDecode pd = make_pixdecode(H, W);
  cudaError_t e = cudaMemsetAsync(start, 0, (size_t)(n + 1) * 4, st);
  if (e != cudaSuccess) return cuda_status(e);
  det_resample_keys_kernel<<<grid_of(n), kSortThreads, 0, st>>>(flow, sb.keys[0], start, B, H, W, pd);
  int rc = after_launch();
  if (rc) return rc;
  const uint32_t* sorted;
  if ((rc = radix_sort(sb, n, (uint32_t)(n - 1), st, &sorted))) return rc;
  if ((rc = exclusive_scan(start, start, n + 1, sb.part, st))) return rc;
  det_resample_gather_kernel<<<grid_of(n), kSortThreads, 0, st>>>(flow, grad_output, sorted, start, grad_input1, B, C, H,
                                                                  W, pd);
  if ((rc = after_launch())) return rc;
  return launch_resample2d_backward_input2(input1, flow, grad_output, grad_input2, B, C, H, W, st);
}
