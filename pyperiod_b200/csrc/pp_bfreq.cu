// pyperiod_b200 -- Periods.best_frequency (pyPeriod/Periods.py:351-398): one fused kernel per round.
//
// A round of the reference is: magnitude spectrum of the residual -> arg-max bin -> p = round(2 * win / bin)
// (:383-386) -> base = project(residual, p, trunc, orth) (:387-389) -> norm, basis out, residual -= base (:390-394).
// The spectrum itself comes from the FFT library (cuFFT through torch: an FFT, not a fold; SURVEY.md 8f); everything
// after it is this kernel: one CTA per window finds the peak bin (first maximum, like np.argmax), derives the
// window's own period, stages the residual, projects it exactly (the bit-exact fold / mean / cofactor chain of
// pp_common.cuh), writes period, norm and basis, and updates the residual in place -- every window with its own
// period in the same launch, no host round trip between rounds.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pyperiod_b200.h"
#include "pp_common.cuh"
#include "pp_host.cuh"

namespace pp {

struct BfPlan {
  int n_even;
  __host__ __device__ size_t off_v() const { return (size_t)n_even * 8; }
  __host__ __device__ size_t off_u() const { return off_v() + (size_t)n_even * 8; }
  __host__ __device__ size_t off_red() const { return off_u() + (size_t)n_even * 8; }
  __host__ __device__ size_t off_bar() const { return off_red() + 2 * kWarps * 8; }
  __host__ __device__ size_t bytes() const { return off_bar() + 32; }
};

size_t bfreq_smem_bytes(int N) {
  BfPlan pl;
  pl.n_even = (N + 1) & ~1;
  return pl.bytes();
}

__global__ void __launch_bounds__(kThreads, 2)
bfreq_round_kernel(double* __restrict__ work, int B, int N, const double* __restrict__ mags, int F, int win, int trunc,
                   int orth, const int32_t* __restrict__ chain_off, const int32_t* __restrict__ chain_q, int table_pmax,
                   uint32_t* __restrict__ periods, double* __restrict__ norms, double* __restrict__ bases, int round,
                   int num, int32_t* __restrict__ status) {
  unsigned char* smem = pp_smem;
  BfPlan pl;
  pl.n_even = (N + 1) & ~1;
  double* xs = reinterpret_cast<double*>(smem);
  double* v = reinterpret_cast<double*>(smem + pl.off_v());
  double* utmp = reinterpret_cast<double*>(smem + pl.off_u());
  double* red = reinterpret_cast<double*>(smem + pl.off_red());
  int* redi = reinterpret_cast<int*>(red + kWarps);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + pl.off_bar());
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  WindowLoader loader;
  loader.init(bar);
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    if (status[b] != PP_STATUS_OK) continue;   // an earlier round failed: the reference has raised by now
    // ---- np.argmax(mags): first index of the maximum; a NaN anywhere wins at its first position
    const double* m = mags + (size_t)b * F;
    double best = -1.0;
    int arg = F;
    for (int i = tid; i < F; i += kThreads) {
      const double a = m[i];
      if (a != a) {
        if (!(best != best) || i < arg) {
          best = a;
          arg = i;
        }
      } else if (!(best != best) && (a > best || (a == best && i < arg))) {
        best = a;
        arg = i;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
      const bool on = ob != ob, bn = best != best;
      const bool take = on ? (!bn || oa < arg) : (!bn && (ob > best || (ob == best && oa < arg)));
      if (take) {
        best = ob;
        arg = oa;
      }
    }
    __syncthreads();
    if (lane == 0) {
      red[wid] = best;
      redi[wid] = arg;
    }
    __syncthreads();
    best = red[0];
    arg = redi[0];
    for (int w = 1; w < kWarps; ++w) {
      const double ob = red[w];
      const int oa = redi[w];
      const bool on = ob != ob, bn = best != best;
      const bool take = on ? (!bn || oa < arg) : (!bn && (ob > best || (ob == best && oa < arg)));
      if (take) {
        best = ob;
        arg = oa;
      }
    }
    __syncthreads();
    if (arg <= 0 || arg >= F) {
      // the DC bin is the peak: p = (2 * win) / 0 -> the reference dies on int(round(inf)) (:386)
      if (tid == 0) status[b] = PP_STATUS_NO_PERIOD;
      continue;
    }
    const int p = (int)rint((2.0 * (double)win) / (double)arg);   // np.round: half to even
    double* wrow = work + (size_t)b * N;
    double* brow = bases ? bases + ((size_t)b * num + round) * N : nullptr;
    double e = 0.0;
    if (p > N) {
      // project() pads the window to ONE row of p samples (:172-176): without truncation the projection is the data
      // itself, with truncation it is a mean over zero rows (nan, :178-184)
      const double nanv = __longlong_as_double(0x7ff8000000000000LL);
      for (int n = tid; n < N; n += kThreads) {
        const double val = trunc ? nanv : wrow[n];
        if (brow) brow[n] = val;
        e = fma(val, val, e);
        wrow[n] = wrow[n] - val;
      }
    } else {
      int clen = 0;
      const int32_t* chain = nullptr;
      if (orth) {
        if (p > table_pmax) {
          if (tid == 0) status[b] = PP_STATUS_GUARD;
          continue;
        }
        chain = chain_q + chain_off[p];
        clen = chain_off[p + 1] - chain_off[p];
      }
      loader.load(xs, wrow, N);
      cta_project_exact<false>(xs, 0, N, p, trunc != 0, chain, clen, v, utmp);
      // ||tile(v)[:N]||^2 = sum_r cnt_r v_r^2 with cnt over all N samples
      const int M = N / p, r0 = N - M * p;
      for (int r = tid; r < p; r += kThreads) e = fma((double)(M + (r < r0 ? 1 : 0)) * v[r], v[r], e);
      if (brow) cta_store_tiled(brow, N, v, p);
      cta_subtract_tiled(xs, N, v, p);
      __syncthreads();
      for (int n = tid; n < N; n += kThreads) wrow[n] = xs[n];
    }
    e = warp_sum(e);
    __syncthreads();
    if (lane == 0) red[wid] = e;
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
      for (int w = 0; w < kWarps; ++w) t += red[w];
      periods[(size_t)b * num + round] = (uint32_t)p;
      norms[(size_t)b * num + round] = sqrt(t) / sqrt((double)N);
    }
    __syncthreads();
  }
}

}  // namespace pp

using namespace pp;

extern "C" {

int pp_best_frequency_round(double* work, int32_t B, int32_t N, const double* mags, int32_t F, int32_t win_size,
                            int32_t trunc, int32_t orth, const int32_t* chain_off, const int32_t* chain_q,
                            int32_t table_pmax, uint32_t* periods, double* norms, double* bases, int32_t round,
                            int32_t num, int32_t* status, void* stream) {
  if (B == 0) return 0;
  if (!work || !mags || !periods || !norms || !status || B < 0 || N < 2 || F < 2 || win_size < 2 || num < 1 || round < 0 ||
      round >= num)
    return fail(-1, "bad best_frequency arguments%s");
  if (orth && (!chain_off || !chain_q)) return fail(-1, "orthogonalize needs the cofactor-chain tables%s");
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  BfPlan pl;
  pl.n_even = (N + 1) & ~1;
  if (int rc = prep_kernel(bfreq_round_kernel, pl.bytes(), f)) return rc;
  bfreq_round_kernel<<<grid_for(f, pl.bytes(), B), kThreads, pl.bytes(), (cudaStream_t)stream>>>(
      work, B, N, mags, F, win_size, trunc, orth, chain_off, chain_q, table_pmax, periods, norms, bases, round, num, status);
  return check_cuda(cudaGetLastError(), "bfreq_round_kernel launch");
}

}  // extern "C"
