// pyperiod_b200 -- the fp64 Ramanujan periodogram in divisor form: O(N + q omega(q)) per (window, period) instead of
// the O(q^2) dense contraction of pp_ramanujan.cu, and the fp64 periodogram of every window whose fused on-chip plan
// does not fit.  Same quantity; see DESIGN.md 5.9 and 5.10.
//
//   c_q(n) = sum_{d | gcd(n, q)} mu(q / d) d   =>   (H S_q)_m = sum_{d | q} mu(q / d) d S_d[m mod d]
//
// With (A_p v)_m = sum_{k < p} v[(m + k q / p) mod q] (the "comb" of prime p: a q/p-periodic vector), the sum is an
// in-place product over the distinct primes of q:
//
//   z = H S_q = (q / rad(q)) prod_{p | q} (p I - A_p) S_q,        norms[q] = (q / phi(q)^2)^2 sum_m cnt_q[m] z_m^2
//
// Per (window, period): fold S_q (rows added in increasing n, one chain per residue, as the sweeps do), then for
// each distinct prime p of q (smallest first, read from the smallest-prime-factor table) the comb sums
// c[j] = sum_{k < p} v[j + k q / p] (k ascending) and v <- p v - c[m mod q / p], then the count-weighted energy.
// All coefficients are small integers.  Every (window, period) result is computed by one warp (on chip) or one CTA
// (global memory) with fixed-order reductions: no floating-point atomics, runs are bit-identical.
//
//   ram_div_chip_kernel    window staged in shared memory once; the CTA's warps take its periods, largest first,
//                          each in a warp-private scratch of qmax + ceil(qmax / 2) doubles (fold + comb sums)
//   ram_div_global_kernel  any N: units (window, period) from a global counter, windows in order and each window's
//                          periods largest first, so the CTAs of the grid fold one window's samples out of L2
//                          together; S_q and the comb sums sit in shared memory when 3 q / 2 doubles fit the
//                          kernel's allotment and in the CTA's slice of the workspace otherwise
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pyperiod_b200.h"
#include "pp_common.cuh"
#include "pp_host.cuh"
#include "pp_sweep.cuh"

namespace pp {
namespace {

constexpr int kDivPad = 32;                      // zero samples after the staged window: fold_range's masked lanes of
                                                 // the last row read up to 31 samples past N
constexpr int kDivGlobalCtas = 296;              // most CTAs the global-memory kernel launches (2 per SM on 148 SMs):
                                                 // bounds the workspace without a device query
constexpr int kDivSmemQ = 8192;                  // largest period the global-memory kernel keeps in shared memory
                                                 // (96 KB of scratch: 2 CTAs per SM)
constexpr size_t kDivCounterBytes = 256;

// doubles of one period's scratch: the fold (q) and the comb sums (q / p <= q / 2), 16-byte aligned
__host__ __device__ inline size_t div_slice(int q) { return ((size_t)q + (size_t)(q + 1) / 2 + 1) & ~(size_t)1; }

// Shared memory of the on-chip kernel: window + pad, kWarps scratches, the period counter.  The launch and
// pp_ramanujan_divisor_fits_on_chip both evaluate this plan.
struct DivisorPlan {
  size_t win_doubles, scratch_doubles;
  size_t dyn;     // dynamic shared memory of the launch
  size_t bytes;   // dyn + the kernel's static shared memory (the window loader's barrier, 128-byte aligned)
};
DivisorPlan divisor_plan(int N, int qmax) {
  DivisorPlan p;
  p.win_doubles = ((size_t)N + kDivPad + 1) & ~(size_t)1;
  p.scratch_doubles = div_slice(qmax);
  p.dyn = (p.win_doubles + (size_t)kWarps * p.scratch_doubles) * 8 + 16;
  p.bytes = p.dyn + 128;
  return p;
}

// doubles of the workspace slice per CTA of the global-memory kernel (0: every period fits its shared memory)
size_t divisor_ws_slices(int qmax) { return qmax > kDivSmemQ ? div_slice(qmax) : 0; }

// ------------------------------------------------------------------------------------------
// the comb factors and the energy, one warp
// ------------------------------------------------------------------------------------------
// v[0 .. q) = S_q on entry (warp-private scratch, c = v + q); returns the norm in every lane
__device__ __forceinline__ double warp_divisor_norm(double* __restrict__ v, int q, int N,
                                                    const int32_t* __restrict__ spf, const int32_t* __restrict__ phi) {
  const int lane = threadIdx.x & 31;
  double* c = v + q;
  int t = q, rad = 1;
  while (t > 1) {
    const int p = __ldg(spf + t);
    const int qp = q / p;
    for (int j = lane; j < qp; j += 32) {
      double s = v[j];
      for (int k = 1; k < p; ++k) s += v[j + k * qp];
      c[j] = s;
    }
    __syncwarp();
    const double pd = (double)p;
    int jm = lane % qp;
    const int step = 32 % qp;
    for (int m = lane; m < q; m += 32) {
      v[m] = pd * v[m] - c[jm];
      jm += step;
      if (jm >= qp) jm -= qp;
    }
    __syncwarp();
    rad *= p;
    do t /= p; while (t % p == 0);
  }
  const int M = N / q, rr = N - M * q;
  const double f = (double)(q / rad);
  double e = 0.0;
  for (int m = lane; m < q; m += 32) {
    const double z = f * v[m];
    e = fma((double)(M + (m < rr ? 1 : 0)) * z, z, e);
  }
  e = warp_sum(e);
  __syncwarp();   // the scratch is reused by the warp's next period
  const double ph = (double)__ldg(phi + q);
  const double scale = (double)q / (ph * ph);
  return scale * scale * e;
}

// ------------------------------------------------------------------------------------------
// on chip: one window per CTA at a time, its periods spread over the warps
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) ram_div_chip_kernel(const double* __restrict__ x, int64_t ldx, int B, int N,
                                                                 int qmin, int qmax, const int32_t* __restrict__ spf,
                                                                 const int32_t* __restrict__ phi,
                                                                 double* __restrict__ norms, int ld_norms,
                                                                 size_t win_doubles, size_t scratch_doubles) {
  double* xs = reinterpret_cast<double*>(pp_smem);
  double* scr = xs + win_doubles + (size_t)(threadIdx.x >> 5) * scratch_doubles;
  int* next = reinterpret_cast<int*>(xs + win_doubles + (size_t)kWarps * scratch_doubles);
  __shared__ uint64_t bar;
  WindowLoader loader;
  loader.init(&bar);
  for (int i = N + threadIdx.x; i < (int)win_doubles; i += kThreads) xs[i] = 0.0;
  const int lane = threadIdx.x & 31;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    __syncthreads();   // every warp is done with the previous window's periods and counter
    if (threadIdx.x == 0) *next = 0;
    loader.load(xs, x + (size_t)b * ldx, N);
    double* out = norms + (size_t)b * ld_norms;
    for (;;) {
      int i = 0;
      if (lane == 0) i = atomicAdd(next, 1);
      const int q = qmax - __shfl_sync(0xffffffffu, i, 0);
      if (q < qmin) break;
      const int M = N / q, rr = N - M * q;
      double T = 0.0, C = 0.0;
      if (rr > 0) fold_range<kPassStore>(xs, q, 0, rr, M + 1, 0, false, 1.0, T, C, scr, scr);
      fold_range<kPassStore>(xs, q, rr, q, M, 0, false, 1.0, T, C, scr, scr);
      __syncwarp();
      const double nrm = warp_divisor_norm(scr, q, N, spf, phi);
      if (lane == 0) out[q] = nrm;
    }
  }
}

// ------------------------------------------------------------------------------------------
// global memory: one (window, period) per CTA at a time
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 2) ram_div_global_kernel(const double* __restrict__ x, int64_t ldx, int N,
                                                                      int qmin, int qmax, long long units,
                                                                      const int32_t* __restrict__ spf,
                                                                      const int32_t* __restrict__ phi,
                                                                      double* __restrict__ norms, int ld_norms,
                                                                      int* counter, double* slices,
                                                                      size_t slice_doubles) {
  __shared__ long long unit;
  __shared__ double red[kWarps];
  double* smem_scr = reinterpret_cast<double*>(pp_smem);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nq = qmax - qmin + 1;
  for (;;) {
    __syncthreads();   // every thread is done with the previous unit's scratch and `unit`
    if (tid == 0) unit = atomicAdd(reinterpret_cast<unsigned long long*>(counter), 1ull);
    __syncthreads();
    const long long u = unit;
    if (u >= units) break;
    const long long b = u / nq;
    const int q = qmax - (int)(u - b * nq);
    double* v = q <= kDivSmemQ ? smem_scr : slices + (size_t)blockIdx.x * slice_doubles;
    double* c = v + q;
    const double* src = x + (size_t)b * ldx;
    // fold: one thread per residue, rows in increasing n
    for (int m = tid; m < q; m += kThreads) {
      double a = __ldg(src + m);
      long long n = m + q;
      for (; n + 3LL * q < N; n += 4LL * q) {
        const double a0 = __ldg(src + n), a1 = __ldg(src + n + q), a2 = __ldg(src + n + 2 * q),
                     a3 = __ldg(src + n + 3 * q);
        a += a0;
        a += a1;
        a += a2;
        a += a3;
      }
      for (; n < N; n += q) a += __ldg(src + n);
      v[m] = a;
    }
    __syncthreads();
    int t = q, rad = 1;
    while (t > 1) {
      const int p = __ldg(spf + t);
      const int qp = q / p;
      for (int j = tid; j < qp; j += kThreads) {
        double s = v[j];
        for (int k = 1; k < p; ++k) s += v[j + k * qp];
        c[j] = s;
      }
      __syncthreads();
      const double pd = (double)p;
      int jm = tid % qp;
      const int step = kThreads % qp;
      for (int m = tid; m < q; m += kThreads) {
        v[m] = pd * v[m] - c[jm];
        jm += step;
        if (jm >= qp) jm -= qp;
      }
      __syncthreads();
      rad *= p;
      do t /= p; while (t % p == 0);
    }
    const int M = N / q, rr = N - M * q;
    const double f = (double)(q / rad);
    double e = 0.0;
    for (int m = tid; m < q; m += kThreads) {
      const double z = f * v[m];
      e = fma((double)(M + (m < rr ? 1 : 0)) * z, z, e);
    }
    e = warp_sum(e);
    if (lane == 0) red[wid] = e;
    __syncthreads();
    if (tid == 0) {
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) s += red[w];
      const double ph = (double)__ldg(phi + q);
      const double scale = (double)q / (ph * ph);
      norms[(size_t)b * ld_norms + q] = scale * scale * s;
    }
  }
}

// CTAs of `kernel` the device holds at once (registers and shared memory), at most `cap` when cap > 0
template <typename K>
long long resident_ctas(K kernel, size_t smem, const DeviceFacts& f, long long cap) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, smem) != cudaSuccess || per_sm < 1)
    per_sm = 1;
  long long g = (long long)per_sm * f.sm_count;
  if (cap > 0 && g > cap) g = cap;
  return g < 1 ? 1 : g;
}

}  // namespace
}  // namespace pp

using namespace pp;

extern "C" {

int pp_ramanujan_divisor_fits_on_chip(int32_t N, int32_t qmin, int32_t qmax, int32_t smem_bytes) {
  if (N < 2 || qmin < 1 || qmax < qmin || qmax > N || smem_bytes < 1) return -1;
  return divisor_plan(N, qmax).bytes <= (size_t)smem_bytes ? 1 : 0;
}

size_t pp_ramanujan_divisor_workspace_bytes(int32_t B, int32_t N, int32_t qmin, int32_t qmax) {
  if (B < 0 || N < 2 || qmin < 1 || qmax < qmin || qmax > N) return 0;
  return kDivCounterBytes + (size_t)kDivGlobalCtas * divisor_ws_slices(qmax) * 8;
}

int pp_ramanujan_norms_divisor(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t qmin, int32_t qmax,
                               const int32_t* spf, const int32_t* phi, int32_t table_qmax, int32_t staging,
                               double* norms, int32_t ld_norms, void* workspace, size_t workspace_bytes,
                               void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (x == nullptr || norms == nullptr || B < 0 || N < 2 || ldx < 1) return fail(-1, "bad window arguments%s");
  if (qmin < 1 || qmax < qmin || qmax > N) return fail(-1, "need 1 <= qmin <= qmax <= N%s");
  if (spf == nullptr || phi == nullptr || table_qmax < qmax) return fail(-1, "spf/phi tables must cover qmax%s");
  if (ld_norms < qmax + 1) return fail(-1, "bad norms leading dimension%s");
  if (staging != PP_STAGING_AUTO && staging != PP_STAGING_SHARED && staging != PP_STAGING_GLOBAL)
    return fail(-1, "unknown staging%s");
  if (workspace == nullptr || workspace_bytes < kDivCounterBytes)
    return fail(-3, "workspace too small (see pp_ramanujan_divisor_workspace_bytes)%s");
  const size_t slice = divisor_ws_slices(qmax);
  const size_t slices_held = slice == 0 ? (size_t)kDivGlobalCtas : (workspace_bytes - kDivCounterBytes) / (slice * 8);
  if (slices_held < 1) return fail(-3, "workspace too small (see pp_ramanujan_divisor_workspace_bytes)%s");
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  const DivisorPlan plan = divisor_plan(N, qmax);
  const bool fits = plan.bytes <= (size_t)f.smem_optin;
  if (staging == PP_STAGING_SHARED && !fits)
    return fail(-1, "the divisor-form plan does not fit in shared memory (use PP_STAGING_GLOBAL or AUTO)%s");
  cudaStream_t st = (cudaStream_t)stream;
  if (staging == PP_STAGING_SHARED || (staging == PP_STAGING_AUTO && fits)) {
    if (int rc = prep_kernel(ram_div_chip_kernel, plan.dyn, f)) return rc;
    const long long grid = resident_ctas(ram_div_chip_kernel, plan.dyn, f, B);
    ram_div_chip_kernel<<<(int)grid, kThreads, plan.dyn, st>>>(x, ldx, B, N, qmin, qmax, spf, phi, norms, ld_norms,
                                                           plan.win_doubles, plan.scratch_doubles);
    return check_cuda(cudaGetLastError(), "ram_div_chip_kernel launch");
  }
  const size_t smem = div_slice(qmax < kDivSmemQ ? qmax : kDivSmemQ) * 8;
  if (int rc = prep_kernel(ram_div_global_kernel, smem, f)) return rc;
  const long long units = (long long)B * (qmax - qmin + 1);
  long long grid = resident_ctas(ram_div_global_kernel, smem, f, 0);
  if (grid > kDivGlobalCtas) grid = kDivGlobalCtas;
  if ((size_t)grid > slices_held) grid = (long long)slices_held;
  if (grid > units) grid = units;
  int* counter = reinterpret_cast<int*>(workspace);
  double* slices = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + kDivCounterBytes);
  if (int rc = check_cuda(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), st), "cudaMemsetAsync")) return rc;
  ram_div_global_kernel<<<(int)grid, kThreads, smem, st>>>(x, ldx, N, qmin, qmax, units, spf, phi, norms, ld_norms,
                                                           counter, slices, slice);
  return check_cuda(cudaGetLastError(), "ram_div_global_kernel launch");
}

}  // extern "C"
