// pyperiod_b200 -- building blocks of the global-memory ("long") paths shared by pp_long.cu (Periods) and
// pp_long_qo.cu (QOPeriods, Muresan): workspace state, the warp-per-candidate sweep, the per-window arg-max, the
// residual loader and the host round helpers.  See pp_long.cu for the design.
#pragma once

#include <cuda_runtime.h>

#include "../../include/pyperiod_b200.h"
#include "pp_common.cuh"
#include "pp_sweep.cuh"
#include "pp_host.cuh"

namespace pp {
namespace {

constexpr int kLongPad = 128;                         // zero samples behind each residual row
constexpr int kLongCtasPerSm = 2;                     // persistent grid of the long kernels

__host__ __device__ inline int long_ldr(int N) { return (N + kLongPad + 31) & ~31; }

// ------------------------------------------------------------------------------------------
// workspace
// ------------------------------------------------------------------------------------------
// Per-window integer state of the round loop (one row of kStateInts per window of the piece).
enum { kActive = 0, kStatus, kFilled, kRepeats, kSweeps, kTies, kNskip, kAction, kSlotId, kCount, kPstart, kStateInts = 16 };
// Per-window double state.
enum { kEres = 0, kDataNorm, kPrev, kOg, kStateDbls = 4 };

struct LongWs {
  int piece = 0, grid = 0, ldr = 0, kld = 0, pv = 0, skw = 0, num = 0;
  double* res = nullptr;     // [piece, ldr]
  double* keys = nullptr;    // [piece, kld]
  double* vu = nullptr;      // [grid, 2 pv]       exact projection vectors of each step CTA
  double* scr = nullptr;     // [grid * kWarps, 2 pv] orthogonalised sweeps / step 2 (orth only)
  double* slots = nullptr;   // [piece, num, pv]   M-best slot bases (one period each)
  double* sd = nullptr;      // [piece, kStateDbls]
  double* norms = nullptr;   // [piece, num]
  int* si = nullptr;         // [piece, kStateInts]
  int* periods = nullptr;    // [piece, num]
  int* slot = nullptr;       // [piece, num]
  uint32_t* skip = nullptr;  // [piece, skw]
  int* list = nullptr;       // [piece] active windows of the round
  int* count = nullptr;      // number of active windows
  int* counter = nullptr;    // unit counter of the sweep
};

// ------------------------------------------------------------------------------------------
// the sweep: one warp per (window, candidate)
// ------------------------------------------------------------------------------------------
// Ranking key of candidate p of the window at xs (global), exactly as warp_period_key computes it from shared memory.
template <int MODE>
__device__ __forceinline__ double long_period_key(const double* xs, int N, int p, bool trunc, int metric, double e_res,
                                                  double data_norm, const int32_t* chain_off, const int32_t* chain_q,
                                                  double* gsS, double* gsV) {
  const int lane = threadIdx.x & 31;
  const int M = N / p, rr = N - M * p;
  const int tail_off = M * p;
  const double m = (double)M;
  double TA = 0.0, TB = 0.0, C = 0.0;
  if (rr > 0) {
    if (MODE == kPassMaxAbs) {
      fold_range<MODE>(xs, p, 0, rr, M + 1, tail_off, false, 0.0, TA, C, gsS, gsV);
    } else {
      fold_range<MODE>(xs, p, 0, rr, trunc ? M : M + 1, tail_off, trunc, trunc ? 1.0 / m : 1.0 / (double)(M + 1), TA,
                       C, gsS, gsV);
    }
  }
  fold_range<(MODE == kPassEnergyTail ? kPassEnergy : MODE)>(xs, p, rr, p, M, tail_off, false, 1.0 / m,
                                                             (MODE == kPassMaxAbs ? TA : TB), C, gsS, gsV);
  if (MODE == kPassMaxAbs) return warp_max(TA);
  double energy, dot;
  if (MODE == kPassStore) {
    __syncwarp();
    warp_orth_chain_approx(gsV, p, N, trunc, chain_q + chain_off[p], chain_off[p + 1] - chain_off[p]);
    double e = 0.0, d = 0.0;
    for (int r = lane; r < p; r += 32) {
      const double v = gsV[r];
      e = fma((double)(M + (r < rr ? 1 : 0)) * v, v, e);
      d = fma(v, gsS[r], d);
    }
    energy = warp_sum(e);
    dot = warp_sum(d);
    __syncwarp();
  } else if (trunc) {
    const double T = TA + TB;
    energy = warp_sum(fma(m, T, TA) / (m * m));
    dot = (MODE == kPassEnergyTail) ? warp_sum((T + C) / m) : energy;
  } else {
    const double w_lo = 1.0 / m, w_diff = 1.0 / (double)(M + 1) - w_lo;
    energy = warp_sum(fma(w_diff, TA, w_lo * (TA + TB)));
    dot = energy;
  }
  if (metric == PP_METRIC_IMPOSED) {
    const double sqrtN = sqrt((double)N);
    const double e_trial = fmax(e_res - 2.0 * dot + energy, 0.0);
    return (sqrt(e_res) / sqrtN - sqrt(e_trial) / sqrtN) / data_norm;  // Periods.py:278-280
  }
  return energy;
}

struct SweepArgs {
  const double* res;
  int ldr, N;
  const int* list;
  const int* count;
  const int* si;          // per-window state: kPstart (first-hit sweeps)
  int pmin, pmax, span;   // candidates of window w: [start, min(start + span - 1, pmax)], start = pmin or kPstart
  int per_window_start;
  int metric, trunc, orth;
  const int32_t* chain_off;
  const int32_t* chain_q;
  const double* sd;       // per-window kEres / kDataNorm (IMPOSED)
  double* keys;
  int kld;
  double* scr;
  int pv;
  int* counter;
};

__global__ void __launch_bounds__(kThreads, kLongCtasPerSm) long_sweep_kernel(SweepArgs a) {
  const int lane = threadIdx.x & 31;
  const long long nact = *a.count;
  const long long total = nact * a.span;
  double* gsS = nullptr;
  double* gsV = nullptr;
  if (a.orth) {
    gsS = a.scr + ((size_t)blockIdx.x * kWarps + (threadIdx.x >> 5)) * 2 * a.pv;
    gsV = gsS + a.pv;
  }
  while (true) {
    long long u = 0;
    if (lane == 0) u = (long long)atomicAdd(reinterpret_cast<unsigned long long*>(a.counter), 1ull);
    u = __shfl_sync(0xffffffffu, u, 0);
    if (u >= total) break;
    const long long j = u / nact;
    const int w = a.list[u - j * nact];
    const int start = a.per_window_start ? a.si[(size_t)w * kStateInts + kPstart] : a.pmin;
    const int p = start + (int)j;
    if (p > a.pmax) continue;
    const double* xs = a.res + (size_t)w * a.ldr;
    double e_res = 0.0, dn = 1.0;
    if (a.metric == PP_METRIC_IMPOSED) {
      e_res = a.sd[(size_t)w * kStateDbls + kEres];
      dn = a.sd[(size_t)w * kStateDbls + kDataNorm];
    }
    const bool trunc = a.trunc != 0;
    double key;
    if (a.metric == PP_METRIC_MAXABS)
      key = long_period_key<kPassMaxAbs>(xs, a.N, p, false, a.metric, 0.0, 1.0, nullptr, nullptr, nullptr, nullptr);
    else if (a.orth)
      key = long_period_key<kPassStore>(xs, a.N, p, trunc, a.metric, e_res, dn, a.chain_off, a.chain_q, gsS, gsV);
    else if (a.metric == PP_METRIC_IMPOSED && trunc)
      key = long_period_key<kPassEnergyTail>(xs, a.N, p, trunc, a.metric, e_res, dn, nullptr, nullptr, nullptr, nullptr);
    else
      key = long_period_key<kPassEnergy>(xs, a.N, p, trunc, a.metric, e_res, dn, nullptr, nullptr, nullptr, nullptr);
    if (lane == 0) a.keys[(size_t)w * a.kld + p] = key;
  }
}

// ------------------------------------------------------------------------------------------
// per-window helpers (one CTA)
// ------------------------------------------------------------------------------------------
struct StepShared {
  double wkey[kWarps];
  int wp[kWarps];
  int misc[8];
  uint32_t mask[kThreads / 32];
  double red[kWarps];
  double wscr[kWarps * 32];
};

// windows of the piece that are still active -> list, count (one warp, ascending order)
__global__ void long_compact_kernel(const int* __restrict__ si, int n, int* __restrict__ list, int* __restrict__ count) {
  const int lane = threadIdx.x & 31;
  int base = 0;
  for (int i0 = 0; i0 < n; i0 += 32) {
    const int i = i0 + lane;
    const bool act = i < n && si[(size_t)i * kStateInts + kActive] != 0;
    const uint32_t m = __ballot_sync(0xffffffffu, act);
    if (act) list[base + __popc(m & ((1u << lane) - 1u))] = i;
    base += __popc(m);
  }
  if (lane == 0) *count = base;
}

// strict '>' arg-max of keys[pmin..pmax] in ascending p (the order of `better`), periods in skip ignored
__device__ Best cta_argmax(const double* keys, int pmin, int pmax, int metric, const uint32_t* skip, StepShared& sh) {
  Best b{0.0, 0};
  for (int p = pmin + threadIdx.x; p <= pmax; p += kThreads) {
    if (skip != nullptr && ((skip[p >> 5] >> (p & 31)) & 1u)) continue;
    const double k = keys[p];
    if (better(metric, k, p, b)) b = Best{k, p};
  }
  b = warp_best(metric, b);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) {
    sh.wkey[threadIdx.x >> 5] = b.key;
    sh.wp[threadIdx.x >> 5] = b.p;
  }
  __syncthreads();
  Best res{0.0, 0};
#pragma unroll
  for (int w = 0; w < kWarps; ++w)
    if (sh.wp[w] != 0 && better(metric, sh.wkey[w], sh.wp[w], res)) res = Best{sh.wkey[w], sh.wp[w]};
  __syncthreads();
  return res;
}

// residual rows of the piece: res[w, 0:N) = x[b0 + w], zero pad behind; sd[w] = sum x^2 and its periodic norm
__global__ void __launch_bounds__(kThreads) long_load_kernel(const double* __restrict__ x, int64_t ldx, int nw, int N,
                                                             double* __restrict__ res, int ldr, double* __restrict__ sd) {
  __shared__ double red[kWarps];
  for (int w = blockIdx.x; w < nw; w += gridDim.x) {
    const double* src = x + (size_t)w * ldx;
    double* dst = res + (size_t)w * ldr;
    for (int n = threadIdx.x; n < ldr; n += kThreads) dst[n] = n < N ? src[n] : 0.0;
    const double e = cta_sum_sq(src, N, red);
    if (threadIdx.x == 0) {
      sd[(size_t)w * kStateDbls + kEres] = e;
      sd[(size_t)w * kStateDbls + kDataNorm] = sqrt(e) / sqrt((double)N);
    }
    __syncthreads();
  }
}

// number of windows still active in the piece: compaction on the device, one 4-byte read-back
static int active_windows(const LongWs& w, int nw, cudaStream_t s, int& nact) {
  long_compact_kernel<<<1, 32, 0, s>>>(w.si, nw, w.list, w.count);
  if (int rc = check_cuda(cudaGetLastError(), "long_compact_kernel launch")) return rc;
  if (int rc = check_cuda(cudaMemcpyAsync(&nact, w.count, sizeof(int), cudaMemcpyDeviceToHost, s), "cudaMemcpyAsync"))
    return rc;
  return check_cuda(cudaStreamSynchronize(s), "cudaStreamSynchronize");
}

static int launch_sweep(const LongWs& w, int N, int pmin, int pmax, int span, bool per_window_start, int metric,
                        int trunc, int orth, const int32_t* chain_off, const int32_t* chain_q, const DeviceFacts& f,
                        cudaStream_t s) {
  if (int rc = check_cuda(cudaMemsetAsync(w.counter, 0, 8, s), "cudaMemsetAsync")) return rc;
  SweepArgs a;
  a.res = w.res;
  a.ldr = w.ldr;
  a.N = N;
  a.list = w.list;
  a.count = w.count;
  a.si = w.si;
  a.pmin = pmin;
  a.pmax = pmax;
  a.span = span;
  a.per_window_start = per_window_start ? 1 : 0;
  a.metric = metric;
  a.trunc = trunc;
  a.orth = orth;
  a.chain_off = chain_off;
  a.chain_q = chain_q;
  a.sd = w.sd;
  a.keys = w.keys;
  a.kld = w.kld;
  a.scr = w.scr;
  a.pv = w.pv;
  a.counter = w.counter;
  (void)f;
  long_sweep_kernel<<<w.grid, kThreads, 0, s>>>(a);
  return check_cuda(cudaGetLastError(), "long_sweep_kernel launch");
}

static int step_grid(const LongWs& w, int nact) { return nact < w.grid ? (nact > 0 ? nact : 1) : w.grid; }

static int check_common_long(const void* x, int64_t ldx, int B, int N) {
  if (x == nullptr) return fail(-1, "x is null%s");
  if (B < 0 || N < 2) return fail(-1, "need B >= 0 and N >= 2%s");
  if (ldx < 1) return fail(-1, "ldx must be >= 1%s");
  return 0;
}

}  // namespace
}  // namespace pp
