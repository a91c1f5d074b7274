// pyperiod_b200 -- device helpers shared by the on-chip (pp_ramanujan.cu) and global-memory (pp_long_ram.cu)
// Ramanujan periodograms: the Ramanujan sum c_q(n), the triangular dictionary layout, cp.async and DMMA.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "pp_common.cuh"

namespace pp {

// c_q(n) = mu(q/g) phi(q) / phi(q/g), g = gcd(n, q): an exact integer (mu / phi: Moebius and totient tables)
__device__ __forceinline__ double ramanujan_sum(int n, int q, const int32_t* __restrict__ mu,
                                                const int32_t* __restrict__ phi) {
  int a = n, b = q;  // gcd(n, q), gcd(0, q) = q
  while (a) {
    const int t = b % a;
    b = a;
    a = t;
  }
  const int g = b, d = q / g;
  return (double)(mu[d] * (phi[q] / phi[d]));
}

// offset of period q in a table of c_q (or of fold rows) for every period from 1: sum_{t<q} t
__host__ __device__ inline size_t cq_offset(int q) { return (size_t)q * (q - 1) / 2; }

// 16-byte asynchronous global -> shared copy; bytes past src_bytes are zero-filled (rows past q, windows past
// the tile)
__device__ __forceinline__ void cp_async_16(void* dst_smem, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst_smem)), "l"(src), "r"(src_bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

__device__ __forceinline__ void dmma_m8n8k4(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c[0]), "+d"(c[1])
               : "d"(a), "d"(b));
}

}  // namespace pp
