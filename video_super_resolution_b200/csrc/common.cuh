// common.cuh -- shared helpers for libvsr_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "../../include/vsr_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libvsr_b200 is written for sm_100a (Blackwell B200) only"
#endif

namespace vsr {

extern std::atomic<uint64_t> g_launch_count;

inline int cuda_status(cudaError_t e) { return e == cudaSuccess ? VSR_OK : VSR_ERR_CUDA_BASE + (int)e; }

// Call right after a <<<>>> launch: counts it and converts a launch error into a VSR code.
inline int after_launch() {
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return cuda_status(cudaGetLastError());
}

inline cudaStream_t as_stream(vsr_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// One-time per-DEVICE setup (function attributes and __constant__ data are per device): the design is one
// process per GPU, but a process that drives several devices must not find the second one unprepared.
struct PerDeviceOnce {
  std::atomic<uint64_t> done{0};          // bit d: device d prepared (devices >= 64 are prepared on every call)
  bool needed(int* dev) {
    if (cudaGetDevice(dev) != cudaSuccess) *dev = 0;
    return *dev >= 64 || !((done.load(std::memory_order_acquire) >> *dev) & 1ull);
  }
  void mark(int dev) {
    if (dev < 64) done.fetch_or(1ull << dev, std::memory_order_release);
  }
};

// Programmatic dependent launch: the next kernel of a stream may start its prologue on SMs the previous
// kernel has already left; it must not touch any buffer an earlier kernel writes or reads before
// griddep_wait(), which returns once every earlier grid has completed and flushed.  Without the launch
// attribute both instructions are no-ops.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

constexpr int kNumSMs = 148;  // B200

__host__ __device__ inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Division by a runtime constant without the ~100-instruction 64-bit divide (ncu: the pixel index ->
// (b, y, x) decode was the bulk of the warp kernels' instructions).  Valid for n < 2^32.
struct FastDiv {
  uint32_t mul, shr, d;
};
inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f;
  f.d = d;
  uint32_t shr = 0;
  while ((1ull << shr) < d) ++shr;
  f.shr = shr;
  f.mul = (uint32_t)((((1ull << 32) * ((1ull << shr) - d)) / d) + 1);
  return f;
}
__device__ __forceinline__ uint32_t fdiv(uint32_t n, const FastDiv& f) {
  return (uint32_t)(((uint64_t)__umulhi(n, f.mul) + n) >> f.shr);
}
// pixel index -> (b, y, x) for a (B, H, W) raster
struct PixDecode {
  FastDiv w, hw;
  uint32_t W, HW;
};
inline PixDecode make_pixdecode(int H, int W) {
  PixDecode d;
  d.w = make_fastdiv((uint32_t)W);
  d.hw = make_fastdiv((uint32_t)H * (uint32_t)W);
  d.W = (uint32_t)W;
  d.HW = (uint32_t)H * (uint32_t)W;
  return d;
}
__device__ __forceinline__ void decode_pix(uint32_t i, const PixDecode& d, int& b, int& y, int& x) {
  const uint32_t bb = fdiv(i, d.hw);
  const uint32_t r = i - bb * d.HW;
  const uint32_t yy = fdiv(r, d.w);
  b = (int)bb;
  y = (int)yy;
  x = (int)(r - yy * d.W);
}

// streaming (read-once) loads / write-once stores: keep them out of L1
__device__ __forceinline__ float2 ldg_stream_f2(const float2* p) {
  float2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_stream_f4(float4* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}

// Stages shared with the deterministic paths (deterministic.cu), launched from the translation unit that owns them.
// The projection's 4-direction hole fill over a list of row words with holes (projection.cu's general path).
int launch_projection_fill(const uint32_t* rowmask, const uint32_t* colmask, const int* n_holewords,
                           const uint32_t* holelist, float* proj, int h, int w, cudaStream_t st);
// Resample2d's gradient w.r.t. the flow (warp.cu), bit-identical to the reference binary.
int launch_resample2d_backward_input2(const float* input1, const float* flow, const float* grad_output,
                                      float* grad_input2, int B, int C, int H, int W, cudaStream_t st);

}  // namespace vsr
