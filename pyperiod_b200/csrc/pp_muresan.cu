// pyperiod_b200 -- Muresan-Parks "equation 3" orthogonal period finder (pyPeriod/QOPeriods.py:1122-1232), batched.
//
// Reference, per window: for every period q in [1, max_p):
//     eq_3(x, q) = (q / N) * (ac(0) + 2 * sum_{l=1}^{M-1} ac(l q)),   M = N // q,  ac(k) = sum_{n < N-k} x[n] x[n+k]
// (:1123-1150, the lag M q is left out), pows[q] = max(eq_3, 0) - sum of pows[f] over the proper divisors f of q
// (:1209-1217, sequential in q), negatives clamped to 0 afterwards, optional division by q, arg-max (:1218-1232).
//
// The autocorrelation sum at multiples of q is the energy of the residue-class fold:
//     sum_r S_q[r]^2 = ac(0) + 2 * sum_{l >= 1, l q < N} ac(l q)
// so eq_3 = (q / N) * (sum_r S_q[r]^2 - 2 ac(M q))  with the last term present only when M q < N: one fold per
// period (the hot primitive of this library) plus one dot product shorter than q.  The divisor recurrence is a
// Moebius inversion, pows[q] = sum_{d | q} mu(q / d) raw[d]: every q is independent, no sequential pass.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pyperiod_b200.h"
#include "pp_common.cuh"
#include "pp_host.cuh"

namespace pp {

__global__ void __launch_bounds__(kThreads, 2)
muresan_kernel(const double* __restrict__ x, int64_t ldx, int B, int N, int max_p, int normalize,
               const int32_t* __restrict__ mu, double* __restrict__ raw_out, double* __restrict__ pows_out,
               int32_t* __restrict__ best_out) {
  unsigned char* smem = pp_smem;
  const int n_even = (N + 1) & ~1;
  double* xs = reinterpret_cast<double*>(smem);
  double* raw = xs + n_even;                                  // [max_p]
  double* pw = raw + ((max_p + 1) & ~1);                      // [max_p]
  double* red = pw + ((max_p + 1) & ~1);                      // [2 * kWarps]
  int* redi = reinterpret_cast<int*>(red + kWarps);
  uint64_t* bar = reinterpret_cast<uint64_t*>(red + 2 * kWarps);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  WindowLoader loader;
  loader.init(bar);
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    loader.load(xs, x + (size_t)b * ldx, N);
    if (tid == 0) {
      raw[0] = 0.0;
      if (raw_out) raw_out[(size_t)b * max_p] = 0.0;
    }
    // ---- raw[q] = max(eq_3(x, q), 0) (raw_out keeps eq_3 itself, which the lag it leaves out can make negative):
    //      one warp per period, lanes over residues, terms in increasing n
    for (int q = 1 + wid; q < max_p; q += kWarps) {
      double e = 0.0;
      for (int r = lane; r < q; r += 32) {
        double s = 0.0;
        for (int n = r; n < N; n += q) s += xs[n];
        e = fma(s, s, e);
      }
      const int lag = (N / q) * q;
      double c = 0.0;
      for (int n = lane; n < N - lag; n += 32) c = fma(xs[n], xs[n + lag], c);
      e = warp_sum(e);
      c = warp_sum(c);
      if (lane == 0) {
        const double v = ((double)q / (double)N) * (e - 2.0 * c);
        raw[q] = fmax(v, 0.0);
        if (raw_out) raw_out[(size_t)b * max_p + q] = v;
      }
    }
    __syncthreads();
    // ---- pows[q] = sum_{d | q} mu(q / d) raw[d], clamp, normalise; arg-max (first maximum)
    double best = -1.0;
    int arg = 0;
    for (int q = tid; q < max_p; q += kThreads) {
      double v = 0.0;
      if (q >= 1) {
        for (int d = 1; d * d <= q; ++d) {
          if (q % d) continue;
          const int d2 = q / d;
          v += (double)mu[d2] * raw[d];
          if (d2 != d) v += (double)mu[d] * raw[d2];
        }
        if (v < 0.0) v = 0.0;
        if (normalize) v = v / (double)q;
      }
      pw[q] = v;
      if (v > best) {
        best = v;
        arg = q;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
      if (ob > best || (ob == best && oa < arg)) {
        best = ob;
        arg = oa;
      }
    }
    if (lane == 0) {
      red[wid] = best;
      redi[wid] = arg;
    }
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < kWarps; ++w)
        if (red[w] > best || (red[w] == best && redi[w] < arg)) {
          best = red[w];
          arg = redi[w];
        }
      // :1226-1232: the strongest period, or 1 when every power is zero
      best_out[b] = arg > 0 ? arg : 1;
    }
    if (pows_out)
      for (int q = tid; q < max_p; q += kThreads) pows_out[(size_t)b * max_p + q] = pw[q];
    __syncthreads();
  }
}

}  // namespace pp

using namespace pp;

size_t pp::muresan_smem_bytes(int N, int max_p) {
  return (size_t)(((N + 1) & ~1) + 2 * ((max_p + 1) & ~1) + 2 * kWarps) * 8 + 64;
}

extern "C" {

int pp_muresan_powers(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t max_p, int32_t normalize,
                      const int32_t* mu, int32_t table_pmax, double* raw, double* pows, int32_t* best, void* stream) {
  if (B == 0) return 0;
  if (!x || !best || !mu || B < 0 || N < 2 || ldx < 1) return fail(-1, "bad arguments%s");
  if (max_p < 2 || max_p > N || table_pmax < max_p - 1) return fail(-1, "need 2 <= max_p <= N and a Moebius table covering max_p - 1%s");
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  const size_t bytes = muresan_smem_bytes(N, max_p);
  if (int rc = prep_kernel(muresan_kernel, bytes, f)) return rc;
  muresan_kernel<<<grid_for(f, bytes, B), kThreads, bytes, (cudaStream_t)stream>>>(x, ldx, B, N, max_p, normalize, mu, raw,
                                                                                  pows, best);
  return check_cuda(cudaGetLastError(), "muresan_kernel launch");
}

}  // extern "C"
