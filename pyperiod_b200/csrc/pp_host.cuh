// pyperiod_b200 -- host-side helpers shared by the translation units of the library.
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>

#include "pp_common.cuh"

namespace pp {

// defined in pp_periods.cu; text retrievable through pp_last_error()
int fail(int code, const char* fmt, const char* a = "");
int check_cuda(cudaError_t e, const char* what);

// shared memory of bfreq_round_kernel for windows of N samples (pp_bfreq.cu)
size_t bfreq_smem_bytes(int N);
// shared memory of muresan_kernel (pp_muresan.cu)
size_t muresan_smem_bytes(int N, int max_p);

// fold modes are per-call arguments (include/pyperiod_b200.h)
static inline int check_fold_mode(int mode) {
  if (mode < 0 || mode > 3) return fail(-1, "unknown fold mode%s");
  return 0;
}

struct DeviceFacts {
  int sm_count = 0, smem_optin = 0, major = 0, minor = 0, clock_khz = 0;
};
static inline int device_facts(DeviceFacts& f) {
  int dev = 0;
  if (int rc = check_cuda(cudaGetDevice(&dev), "cudaGetDevice")) return rc;
  cudaDeviceGetAttribute(&f.sm_count, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(&f.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  cudaDeviceGetAttribute(&f.major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&f.minor, cudaDevAttrComputeCapabilityMinor, dev);
  cudaDeviceGetAttribute(&f.clock_khz, cudaDevAttrClockRate, dev);
  return 0;
}

// L2 cache of the current device: the global-memory paths size their pieces from it
static inline int l2_bytes() {
  int dev = 0, l2 = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev);
  return l2 > 0 ? l2 : (64 << 20);
}

// persistent grid: CTAs per SM limited by shared memory (and by kCtasPerSm through registers)
static inline int grid_for(const DeviceFacts& f, size_t smem_bytes, int B, int max_per_sm = kCtasPerSm) {
  int per_sm = (int)((size_t)(f.smem_optin + 1024) / (smem_bytes + 1024));
  if (per_sm > max_per_sm) per_sm = max_per_sm;
  if (per_sm < 1) per_sm = 1;
  int g = f.sm_count * per_sm;
  if (B > 0 && g > B) g = B;
  return g < 1 ? 1 : g;
}

template <typename K>
static inline int prep_kernel(K kernel, size_t smem_bytes, const DeviceFacts& f) {
  if (smem_bytes > (size_t)f.smem_optin)
    return fail(-2, "window does not fit in shared memory for on-chip staging%s");
  return check_cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes),
                    "cudaFuncSetAttribute");
}

// bump allocator over the caller-owned workspace (256-byte aligned pieces)
static inline double* carve(void* ws, size_t ws_bytes, size_t& off, size_t bytes) {
  off = (off + 255) & ~(size_t)255;
  if (ws == nullptr || off + bytes > ws_bytes) return nullptr;
  double* p = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + off);
  off += bytes;
  return p;
}

// global window counter of a WindowQueue, zeroed on `stream`; nullptr (static stride) when the workspace has no room
static inline int* carve_window_counter(void* ws, size_t ws_bytes, size_t& off, cudaStream_t stream) {
  double* p = carve(ws, ws_bytes, off, 256);
  if (p == nullptr) return nullptr;
  if (cudaMemsetAsync(p, 0, sizeof(int), stream) != cudaSuccess) return nullptr;
  return reinterpret_cast<int*>(p);
}

}  // namespace pp
