// api.cu -- library identification, error strings and launch accounting.
#include "common.cuh"

#include <stdio.h>

namespace vsr {
std::atomic<uint64_t> g_launch_count{0};
}

extern "C" const char* vsr_version(void) { return "vsr_b200 0.1 (sm_100a)"; }

extern "C" uint64_t vsr_launch_count(void) { return vsr::g_launch_count.load(std::memory_order_relaxed); }

extern "C" void vsr_launch_count_reset(void) { vsr::g_launch_count.store(0, std::memory_order_relaxed); }

extern "C" const char* vsr_error_string(int code) {
  static thread_local char buf[160];
  switch (code) {
    case VSR_OK: return "ok";
    case VSR_ERR_INVALID_ARG: return "invalid argument (null pointer, non-positive size, misaligned buffer)";
    case VSR_ERR_UNSUPPORTED: return "unsupported shape / option";
    case VSR_ERR_WORKSPACE: return "workspace too small";
    case VSR_ERR_STATE: return "plan not ready (weights/workspace not bound)";
    default: break;
  }
  if (code >= VSR_ERR_CUDA_BASE) {
    snprintf(buf, sizeof(buf), "CUDA error %d: %s", code - VSR_ERR_CUDA_BASE,
             cudaGetErrorString((cudaError_t)(code - VSR_ERR_CUDA_BASE)));
    return buf;
  }
  snprintf(buf, sizeof(buf), "unknown vsr error %d", code);
  return buf;
}
