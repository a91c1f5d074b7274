// pyperiod_b200 -- the global-memory ("long") path of the `Periods` family: windows whose on-chip plan does not fit
// the shared memory of one CTA (pp_fits_on_chip).  Same results contract as the on-chip kernels of pp_periods.cu /
// pp_bfreq.cu, which stay untouched.
//
// Layout.  Batches run in pieces of windows.  Each window of a piece has its residual copied into the workspace
// (`res[piece, ldr]`, zero padded: the partial register tiles of the fold read up to 63 samples past N); the caller's
// input is never written.  The piece is sized so its residuals stay within half of the L2 cache.
//
// Rounds, driven by the host on the caller's stream:
//   sweep   long_sweep_kernel: one unit per (active window, candidate p), handed out to warps by a global counter
//           over the whole GPU.  A warp folds its candidate from the residual with the register tiles of the direct
//           fold (pp_sweep.cuh fold_range: rows in increasing n, 256-byte row segments) and writes keys[w, p] with
//           the on-chip direct fold's reduction order -- no floating-point atomics, so results are run-to-run
//           identical, and MAXABS keys are the reference's exact sequential sums.
//   step    one CTA per active window: arg-max (strict '>', lowest p on ties), the near-tie audit of NORM / GAMMA
//           sweeps, the exact projection (cta_project_exact on global pointers), bookkeeping and the residual update.
//   The host reads the number of windows still active (4 bytes, cudaMemcpyAsync) once per round and stops at 0.
#include <cuda_runtime.h>
#include <string.h>

#include "../../include/pyperiod_b200.h"
#include "pp_common.cuh"
#include "pp_sweep.cuh"
#include "pp_host.cuh"
#include "pp_long.cuh"

namespace pp {
namespace {

constexpr size_t kOrthScratchBudget = 512ull << 20;   // per-warp p-vectors of orthogonalised sweeps
constexpr int kS2lMinChunk = 32;                      // small-to-large: candidates per window and round, at least
constexpr int kS2lMaxChunk = 4096;

// Sizes (base == nullptr) or carves the workspace of one long-path call.  Returns the bytes needed.
static size_t long_layout(int algo, int B, int N, int pmax, int num, int orth, const DeviceFacts& f, void* base,
                          size_t bytes, LongWs& w) {
  w.ldr = long_ldr(N);
  w.pv = (pmax + 2) & ~1;
  w.kld = pmax + 1;
  w.skw = (pmax + 32) / 32;
  w.num = algo == PP_ALGO_MBEST ? num : 0;
  const size_t res_bytes = (size_t)w.ldr * 8;
  size_t piece = (size_t)l2_bytes() / 2 / res_bytes;
  if (piece < 1) piece = 1;
  if (piece > (size_t)B) piece = B > 0 ? (size_t)B : 1;
  w.piece = (int)piece;
  int grid = f.sm_count * kLongCtasPerSm;
  if (orth) {
    const size_t per_cta = (size_t)kWarps * 2 * w.pv * 8;
    const size_t cap = kOrthScratchBudget / per_cta;
    if ((size_t)grid > cap) grid = cap < 1 ? 1 : (int)cap;
  }
  if (algo == PP_ALGO_PROJECT && grid > B) grid = B > 0 ? B : 1;
  w.grid = grid;
  const bool rounds = algo != PP_ALGO_PROJECT && algo != PP_ALGO_BFREQ;
  size_t off = 0;
  auto take = [&](size_t n) -> void* {
    off = (off + 255) & ~(size_t)255;
    void* p = (base != nullptr && off + n <= bytes) ? (void*)((char*)base + off) : nullptr;
    off += n;
    return p;
  };
  w.vu = (double*)take((size_t)grid * 2 * w.pv * 8);
  if (rounds) {
    w.res = (double*)take(piece * res_bytes);
    w.keys = (double*)take(piece * (size_t)w.kld * 8);
    w.scr = orth ? (double*)take((size_t)grid * kWarps * 2 * w.pv * 8) : nullptr;
    w.sd = (double*)take(piece * kStateDbls * 8);
    w.si = (int*)take(piece * kStateInts * 4);
    w.list = (int*)take(piece * 4);
    w.count = (int*)take(256);
    w.counter = (int*)take(256);
    if (algo == PP_ALGO_MBEST) {
      w.slots = (double*)take(piece * (size_t)num * w.pv * 8);
      w.norms = (double*)take(piece * (size_t)num * 8);
      w.periods = (int*)take(piece * (size_t)num * 4);
      w.slot = (int*)take(piece * (size_t)num * 4);
      w.skip = (uint32_t*)take(piece * (size_t)w.skw * 4);
    }
  }
  return off + 256;
}

// cta_canonical_value (pp_sweep.cuh) on a window in global memory
__device__ double long_canonical_value(const double* xs, int N, int p, int metric, bool trunc, bool orth,
                                       const int32_t* chain_off, const int32_t* chain_q, double* v, double* u,
                                       StepShared& sh) {
  const int clen = orth ? chain_off[p + 1] - chain_off[p] : 0;
  __syncthreads();
  cta_project_exact<false>(xs, 0, N, p, trunc, orth ? chain_q + chain_off[p] : nullptr, clen, v, u);
  double a = 0.0;
  int r = threadIdx.x % p;
  const int step = kThreads % p;
  for (int n = threadIdx.x; n < N; n += kThreads) {
    const double b = v[r];
    a = fma(b, b, a);
    r += step;
    if (r >= p) r -= p;
  }
  a = warp_sum(a);
  if ((threadIdx.x & 31) == 0) sh.wkey[threadIdx.x >> 5] = a;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < kWarps; ++w) t += sh.wkey[w];
  __syncthreads();
  return key_to_value(metric, t, p, sqrt((double)N));
}

// Winner of a NORM / GAMMA sweep with the near-tie audit of cta_sweep: every candidate whose key can reach the best
// within the rounding bound is re-evaluated the reference's way and ranked by value, strict '>' in ascending p.
// *nnom = candidates inside the bound (1 = a clear winner).
__device__ SweepResult cta_pick_audited(const double* keys, const double* xs, int N, int pmin, int pmax, int metric,
                                        bool trunc, bool orth, double e_bound, const uint32_t* skip,
                                        const int32_t* chain_off, const int32_t* chain_q, double* v, double* u,
                                        StepShared& sh, int* nnom_out) {
  const Best res = cta_argmax(keys, pmin, pmax, metric, skip, sh);
  SweepResult out{0.0, res.p};
  int nnom = 0;
  if (res.p != 0) {
    out.val = key_to_value(metric, res.key, res.p, sqrt((double)N));
    const bool gam = metric == PP_METRIC_GAMMA;
    const double lo_best = res.key - tie_tol(N, res.p, e_bound);
    auto nominated = [&](int p) {
      if (p > pmax) return false;
      if (skip != nullptr && ((skip[p >> 5] >> (p & 31)) & 1u)) return false;
      const double hi = keys[p] + tie_tol(N, p, e_bound);
      return gam ? hi * (double)res.p >= lo_best * (double)p : hi >= lo_best;
    };
    for (int base = pmin; base <= pmax; base += kThreads) nnom += __syncthreads_count(nominated(base + threadIdx.x));
    if (nnom > 1) {
      double best_v = 0.0;
      int best_p = 0;
      for (int base = pmin; base <= pmax; base += kThreads) {
        const bool in = nominated(base + threadIdx.x);
        const uint32_t m = __ballot_sync(0xffffffffu, in);
        if ((threadIdx.x & 31) == 0) sh.mask[threadIdx.x >> 5] = m;
        __syncthreads();
        for (int wd = 0; wd < kWarps; ++wd) {
          uint32_t bits = sh.mask[wd];  // uniform
          while (bits) {
            const int p = base + wd * 32 + __ffs(bits) - 1;
            bits &= bits - 1;
            const double val = long_canonical_value(xs, N, p, metric, trunc, orth, chain_off, chain_q, v, u, sh);
            if (val > best_v) {
              best_v = val;
              best_p = p;
            }
          }
        }
        __syncthreads();
      }
      out.p = best_p;
      out.val = best_v;
    }
  }
  *nnom_out = nnom;
  return out;
}

// ------------------------------------------------------------------------------------------
// project
// ------------------------------------------------------------------------------------------
struct ChainArgL {
  int32_t q[16];
  int32_t len;
};

__global__ void __launch_bounds__(kThreads) long_project_kernel(const double* __restrict__ x, int64_t ldx, int B, int N,
                                                                int p, int trunc, ChainArgL chain, double* __restrict__ out,
                                                                int64_t ldo, int out_len, double* __restrict__ vu, int pv) {
  __shared__ int32_t s_chain[16];
  if (threadIdx.x < 16) s_chain[threadIdx.x] = chain.q[threadIdx.x];
  __syncthreads();
  double* v = vu + (size_t)blockIdx.x * 2 * pv;
  double* u = v + pv;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    cta_project_exact<false>(x + (size_t)b * ldx, 0, N, p, trunc != 0, s_chain, chain.len, v, u);
    cta_store_tiled(out + (size_t)b * ldo, out_len, v, p);
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// sweep (one round): metrics, arg-max, near-tie audit
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) long_sweep_step_kernel(LongWs w, int N, int pmin, int pmax, int metric,
                                                                   int trunc, int orth, const int32_t* chain_off,
                                                                   const int32_t* chain_q, double* __restrict__ metric_out,
                                                                   int32_t* __restrict__ best_p,
                                                                   double* __restrict__ best_val, int b0) {
  __shared__ StepShared sh;
  double* v = w.vu + (size_t)blockIdx.x * 2 * w.pv;
  double* u = v + w.pv;
  const double sqrtN = sqrt((double)N);
  const int nact = *w.count;
  for (int i = blockIdx.x; i < nact; i += gridDim.x) {
    const int wi = w.list[i];
    const int b = b0 + wi;
    const double* keys = w.keys + (size_t)wi * w.kld;
    const double* xs = w.res + (size_t)wi * w.ldr;
    if (metric_out != nullptr)
      for (int p = pmin + threadIdx.x; p <= pmax; p += kThreads)
        metric_out[(size_t)b * (pmax + 1) + p] = key_to_value(metric, keys[p], p, sqrtN);
    SweepResult r;
    if (metric == PP_METRIC_NORM || metric == PP_METRIC_GAMMA) {
      int nnom = 0;
      r = cta_pick_audited(keys, xs, N, pmin, pmax, metric, trunc != 0, orth != 0, w.sd[(size_t)wi * kStateDbls + kEres],
                           nullptr, chain_off, chain_q, v, u, sh, &nnom);
    } else {
      const Best res = cta_argmax(keys, pmin, pmax, metric, nullptr, sh);
      r = SweepResult{res.p != 0 ? key_to_value(metric, res.key, res.p, sqrtN) : 0.0, res.p};
    }
    if (threadIdx.x == 0) {
      best_p[b] = r.p;
      best_val[b] = r.val;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// M-best
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) long_mbest_init_kernel(LongWs w, int nw, int num) {
  for (int wi = blockIdx.x; wi < nw; wi += gridDim.x) {
    int* si = w.si + (size_t)wi * kStateInts;
    if (threadIdx.x < kStateInts) si[threadIdx.x] = threadIdx.x == kActive ? 1 : 0;
    for (int i = threadIdx.x; i < num; i += kThreads) {
      w.periods[(size_t)wi * num + i] = 0;
      w.norms[(size_t)wi * num + i] = 0.0;
      w.slot[(size_t)wi * num + i] = i;
    }
    for (int i = threadIdx.x; i < w.skw; i += kThreads) w.skip[(size_t)wi * w.skw + i] = 0u;
  }
}

// step 1 of M-best for one sweep (Periods.py:494-537): winner, slot bookkeeping, residual update
__global__ void __launch_bounds__(kThreads) long_mbest_step_kernel(LongWs w, int N, int num, int pmin, int pmax, int gamma,
                                                                   int trunc_i, int orth_i, const int32_t* chain_off,
                                                                   const int32_t* chain_q, int guard) {
  __shared__ StepShared sh;
  const bool trunc = trunc_i != 0, orth = orth_i != 0;
  const int metric = gamma ? PP_METRIC_GAMMA : PP_METRIC_NORM;
  double* v = w.vu + (size_t)blockIdx.x * 2 * w.pv;
  double* u = v + w.pv;
  const int nact = *w.count;
  for (int i = blockIdx.x; i < nact; i += gridDim.x) {
    const int wi = w.list[i];
    int* si = w.si + (size_t)wi * kStateInts;
    int* periods = w.periods + (size_t)wi * num;
    double* norms = w.norms + (size_t)wi * num;
    int* slot = w.slot + (size_t)wi * num;
    uint32_t* skip = w.skip + (size_t)wi * w.skw;
    double* xs = w.res + (size_t)wi * w.ldr;
    int nnom = 0;
    const SweepResult top = cta_pick_audited(w.keys + (size_t)wi * w.kld, xs, N, pmin, pmax, metric, trunc, orth,
                                             w.sd[(size_t)wi * kStateDbls + kEres], si[kNskip] > 0 ? skip : nullptr,
                                             chain_off, chain_q, v, u, sh, &nnom);
    const int sweeps = si[kSweeps] + 1;
    __syncthreads();
    if (threadIdx.x == 0) {
      si[kSweeps] = sweeps;
      if (nnom > 1) si[kTies] += 1;
    }
    if (top.p == 0 || sweeps > guard) {
      if (threadIdx.x == 0) {
        si[kStatus] = top.p == 0 ? PP_STATUS_NO_PERIOD : PP_STATUS_GUARD;
        si[kActive] = 0;
      }
      __syncthreads();
      continue;
    }
    const int clen = orth ? chain_off[top.p + 1] - chain_off[top.p] : 0;
    cta_project_exact<false>(xs, 0, N, top.p, trunc, orth ? chain_q + chain_off[top.p] : nullptr, clen, v, u);
    if (threadIdx.x == 0) {
      int found = -1;
      for (int k = 0; k < num; ++k)
        if (periods[k] == top.p) found = k;
      if (found >= 0 && si[kRepeats] < 10) {   // strengthen an existing slot (:518-524)
        norms[found] += top.val;
        si[kRepeats] += 1;
        sh.misc[0] = 0;
        sh.misc[1] = slot[found];
      } else if (found >= 0) {                 // blacklist it (:525-529)
        skip[top.p >> 5] |= 1u << (top.p & 31);
        si[kNskip] += 1;
        si[kRepeats] = 0;
        sh.misc[0] = 1;
      } else {                                 // new slot (:530-535)
        const int k = si[kFilled];
        periods[k] = top.p;
        norms[k] = top.val;
        si[kFilled] = k + 1;
        si[kRepeats] = 0;
        sh.misc[0] = 2;
        sh.misc[1] = slot[k];
      }
      if (si[kFilled] >= num) si[kActive] = 0;
    }
    __syncthreads();
    const int action = sh.misc[0];
    if (action != 1) {
      double* sl = w.slots + ((size_t)wi * num + sh.misc[1]) * w.pv;
      if (action == 0) {
        for (int r = threadIdx.x; r < top.p; r += kThreads) sl[r] += v[r];
      } else {
        for (int r = threadIdx.x; r < top.p; r += kThreads) sl[r] = v[r];
      }
    }
    cta_subtract_tiled(xs, N, v, top.p);  // always (:537)
    __syncthreads();
  }
}

// Norm of the projection of a P-periodic slot basis onto divisor f, by one warp (warp_slot_factor_norm of
// pp_periods.cu on global pointers).
__device__ __forceinline__ double long_slot_factor_norm(const double* slot, int P, int f, int N, bool trunc, bool orth,
                                                        const int32_t* chain_off, const int32_t* chain_q, double* scr,
                                                        double sqrtN, double* wscr) {
  const int lane = threadIdx.x & 31;
  const int t = P / f;
  const int Mf = N / f, r0f = N - Mf * f;
  const double rcp_lo = 1.0 / (double)Mf, rcp_hi = 1.0 / (double)(Mf + 1);
  double e = 0.0;
  if (f < 32) {
    const int g = 32 / f;
    const int r = lane % f, grp = lane / f;
    const int K = trunc ? Mf : (Mf + (r < r0f ? 1 : 0));
    const int base = K / t, rem = K - base * t;
    double s = 0.0;
    if (grp < g)
      for (int j = grp; j < t; j += g) s = fma((double)(base + (j < rem ? 1 : 0)), slot[r + j * f], s);
    wscr[lane] = s;
    __syncwarp();
    if (lane < f) {
      double tot = wscr[lane];
      for (int k = 1; k < g; ++k) tot += wscr[lane + k * f];
      const double mean = tot * (K == Mf ? rcp_lo : rcp_hi);
      if (orth) scr[lane] = mean;
      else e = (double)(Mf + (lane < r0f ? 1 : 0)) * mean * mean;
    }
    __syncwarp();
  } else {
    for (int r = lane; r < f; r += 32) {
      const int K = trunc ? Mf : (Mf + (r < r0f ? 1 : 0));
      const int base = K / t, rem = K - base * t;
      double s = 0.0;
      for (int j = 0; j < t; ++j) s = fma((double)(base + (j < rem ? 1 : 0)), slot[r + j * f], s);
      const double mean = s * (K == Mf ? rcp_lo : rcp_hi);
      if (orth) scr[r] = mean;
      else e = fma((double)(Mf + (r < r0f ? 1 : 0)) * mean, mean, e);
    }
  }
  if (orth) {
    __syncwarp();
    warp_orth_chain_approx(scr, f, N, trunc, chain_q + chain_off[f], chain_off[f + 1] - chain_off[f]);
    for (int r = lane; r < f; r += 32) {
      const double vv = scr[r];
      e = fma((double)(Mf + (r < r0f ? 1 : 0)) * vv, vv, e);
    }
    __syncwarp();
  }
  return sqrt(warp_sum(e)) / sqrtN;
}

// step 2 of M-best (Periods.py:540-598, one pass) and the outputs; one CTA per window of the piece.  The divisor
// lists are read from the tables in place: no cap on their length.
__global__ void __launch_bounds__(kThreads) long_mbest_final_kernel(
    LongWs w, int nw, int N, int num, int pmax, int gamma, int trunc_i, int orth_i, const int32_t* chain_off,
    const int32_t* chain_q, const int32_t* fac_off, const int32_t* fac, int b0, uint32_t* __restrict__ periods_out,
    double* __restrict__ powers_out, double* __restrict__ bases_out, int32_t* __restrict__ sweeps_out,
    int32_t* __restrict__ near_ties_out, int32_t* __restrict__ status_out) {
  __shared__ StepShared sh;
  const bool trunc = trunc_i != 0, orth = orth_i != 0;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const double sqrtN = sqrt((double)N);
  double* v = w.vu + (size_t)blockIdx.x * 2 * w.pv;
  double* u = v + w.pv;
  double* my_scr = orth ? w.scr + ((size_t)blockIdx.x * kWarps + wid) * 2 * w.pv : nullptr;
  for (int wi = blockIdx.x; wi < nw; wi += gridDim.x) {
    const int b = b0 + wi;
    int* si = w.si + (size_t)wi * kStateInts;
    int* periods = w.periods + (size_t)wi * num;
    double* norms = w.norms + (size_t)wi * num;
    int* slot = w.slot + (size_t)wi * num;
    double* my_slots = w.slots + (size_t)wi * num * w.pv;
    double* sl_s = w.res + (size_t)wi * w.ldr;   // the residual is dead after step 1
    __syncthreads();
    if (threadIdx.x == 0) sh.misc[4] = si[kStatus];
    __syncthreads();
    if (sh.misc[4] == PP_STATUS_OK) {
      const double stale_div = sqrt((double)pmax);  // gamma norms divide by sqrt(max_length) (:559,:572)
      int i = 0, changes = 0;
      while (i < num) {
        const int P = periods[i];
        const double* sl = my_slots + (size_t)slot[i] * w.pv;
        const int f0 = fac_off[P], nf = fac_off[P + 1] - f0;
        if (changes > 64 * num) {
          if (threadIdx.x == 0) sh.misc[4] = PP_STATUS_GUARD;
          __syncthreads();
          break;
        }
        __syncthreads();
        for (int r = threadIdx.x; r < P; r += kThreads) sl_s[r] = sl[r];
        __syncthreads();
        double w_top = 0.0;
        int w_fi = -1;
        for (int fi = wid; fi < nf; fi += kWarps) {
          const int f = fac[f0 + fi];
          double val = long_slot_factor_norm(sl_s, P, f, N, trunc, orth, chain_off, chain_q, my_scr, sqrtN,
                                             sh.wscr + wid * 32);
          if (gamma) val = val / stale_div;
          if (val > w_top) {
            w_top = val;
            w_fi = fi;
          }
          if (fi == nf - 1 && lane == 0) sh.red[0] = val;  // norm of the LAST factor's projection (:570-572)
        }
        if (lane == 0) {
          sh.wkey[wid] = w_top;
          sh.wp[wid] = w_fi;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
          double top = 0.0;
          int top_fi = -1;
          for (int q = 0; q < kWarps; ++q)
            if (sh.wp[q] >= 0 && (sh.wkey[q] > top || (sh.wkey[q] == top && top_fi >= 0 && sh.wp[q] < top_fi))) {
              top = sh.wkey[q];
              top_fi = sh.wp[q];
            }
          const int top_f = top_fi >= 0 ? fac[f0 + top_fi] : 0;
          int decision = 0;
          if (top_f != 0) {
            bool present = false;
            double floor_n = norms[0];
            const double n_weak = sh.red[0], n_last = norms[num - 1], n_i = norms[i];
            for (int k = 0; k < num; ++k) {
              present |= (periods[k] == top_f);
              floor_n = fmin(floor_n, norms[k]);
            }
            if (!present) {
              const double n_strong = top;
              if ((n_weak + n_strong) > (n_last + n_i) && n_weak > floor_n && n_strong > floor_n) {
                decision = 1;
                const int freed = slot[num - 1];
                for (int k = num - 1; k > i; --k) {
                  periods[k] = periods[k - 1];
                  norms[k] = norms[k - 1];
                  slot[k] = slot[k - 1];
                }
                if (i + 1 < num) norms[i + 1] = n_weak;
                periods[i] = top_f;
                norms[i] = n_strong;
                slot[i] = freed;
                sh.misc[3] = freed;
              }
            }
          }
          sh.misc[5] = decision;
          sh.misc[6] = top_f;
        }
        __syncthreads();
        if (sh.misc[5]) {
          const int f = sh.misc[6];
          const int clen = orth ? chain_off[f + 1] - chain_off[f] : 0;
          cta_project_exact<true>(sl_s, P, N, f, trunc, orth ? chain_q + chain_off[f] : nullptr, clen, v, u);
          double* old_sl = const_cast<double*>(sl);
          double* new_sl = my_slots + (size_t)sh.misc[3] * w.pv;
          if (i + 1 < num) {
            int rq = threadIdx.x % f;
            const int step = kThreads % f;
            for (int r = threadIdx.x; r < P; r += kThreads) {
              old_sl[r] = sl_s[r] - v[rq];
              rq += step;
              if (rq >= f) rq -= f;
            }
          }
          __syncthreads();
          for (int r = threadIdx.x; r < f; r += kThreads) new_sl[r] = v[r];
          ++changes;
          __syncthreads();
        } else {
          ++i;
        }
      }
    }
    __syncthreads();
    const int status = sh.misc[4];
    const double data_norm = w.sd[(size_t)wi * kStateDbls + kDataNorm];
    for (int k = threadIdx.x; k < num; k += kThreads) {
      const bool ok = status == PP_STATUS_OK;
      periods_out[(size_t)b * num + k] = ok ? (uint32_t)periods[k] : 0u;
      powers_out[(size_t)b * num + k] = ok ? norms[k] / data_norm : 0.0;
    }
    if (threadIdx.x == 0) {
      status_out[b] = status;
      if (sweeps_out) sweeps_out[b] = si[kSweeps];
      if (near_ties_out) near_ties_out[b] = si[kTies];
    }
    if (bases_out != nullptr) {
      for (int k = 0; k < num; ++k) {
        double* dst = bases_out + ((size_t)b * num + k) * N;
        const int P = periods[k];
        if (status == PP_STATUS_OK && P > 0) cta_store_tiled(dst, N, my_slots + (size_t)slot[k] * w.pv, P);
        else
          for (int n = threadIdx.x; n < N; n += kThreads) __stcs(dst + n, 0.0);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// small-to-large
// ------------------------------------------------------------------------------------------
// every window of the piece active, first-hit sweeps start at p = 2
__global__ void __launch_bounds__(kThreads) long_activate_kernel(LongWs w, int nw) {
  for (int wi = blockIdx.x; wi < nw; wi += gridDim.x) {
    int* si = w.si + (size_t)wi * kStateInts;
    if (threadIdx.x < kStateInts) si[threadIdx.x] = threadIdx.x == kActive ? 1 : (threadIdx.x == kPstart ? 2 : 0);
  }
}

// first hit of this window's chunk [pstart, pstart + span): accept, project, subtract, restart at p + 1
// (Periods.py:273-286); no hit: the next chunk
__global__ void __launch_bounds__(kThreads) long_s2l_step_kernel(LongWs w, int N, double thresh, int n_periods, int span,
                                                                 int trunc_i, int orth_i, const int32_t* chain_off,
                                                                 const int32_t* chain_q, int kmax, int b0,
                                                                 uint32_t* __restrict__ periods_out,
                                                                 double* __restrict__ powers_out,
                                                                 double* __restrict__ bases_out) {
  __shared__ StepShared sh;
  const bool trunc = trunc_i != 0, orth = orth_i != 0;
  double* v = w.vu + (size_t)blockIdx.x * 2 * w.pv;
  double* u = v + w.pv;
  const int nact = *w.count;
  for (int i = blockIdx.x; i < nact; i += gridDim.x) {
    const int wi = w.list[i];
    const int b = b0 + wi;
    int* si = w.si + (size_t)wi * kStateInts;
    double* sd = w.sd + (size_t)wi * kStateDbls;
    const double* keys = w.keys + (size_t)wi * w.kld;
    double* xs = w.res + (size_t)wi * w.ldr;
    const int ps = si[kPstart];
    const int last = min(ps + span - 1, n_periods);
    __syncthreads();
    if (threadIdx.x == 0) sh.misc[0] = 0x7fffffff;
    __syncthreads();
    for (int p = ps + threadIdx.x; p <= last; p += kThreads)
      if (keys[p] > thresh) atomicMin(&sh.misc[0], p);
    __syncthreads();
    const int hit = sh.misc[0];
    if (hit == 0x7fffffff) {
      if (threadIdx.x == 0) {
        si[kPstart] = last + 1;
        if (last + 1 > n_periods) si[kActive] = 0;
      }
      continue;
    }
    const double val = keys[hit];
    const int clen = orth ? chain_off[hit + 1] - chain_off[hit] : 0;
    cta_project_exact<false>(xs, 0, N, hit, trunc, orth ? chain_q + chain_off[hit] : nullptr, clen, v, u);
    cta_subtract_tiled(xs, N, v, hit);
    const int count = si[kCount];
    if (count < kmax) {
      if (threadIdx.x == 0) {
        periods_out[(size_t)b * kmax + count] = (uint32_t)hit;
        powers_out[(size_t)b * kmax + count] = val;
      }
      if (bases_out) cta_store_tiled(bases_out + ((size_t)b * kmax + count) * N, N, v, hit);
    }
    __syncthreads();
    const double e_now = cta_sum_sq(xs, N, sh.red);
    if (threadIdx.x == 0) {
      si[kCount] = count + 1;
      sd[kEres] = e_now;
      si[kPstart] = hit + 1;
      if (hit + 1 > n_periods) si[kActive] = 0;
    }
    __syncthreads();
  }
}

__global__ void long_s2l_final_kernel(const int* __restrict__ si, int nw, int kmax, int b0, uint32_t* __restrict__ periods_out,
                                      double* __restrict__ powers_out, int32_t* __restrict__ count_out,
                                      int32_t* __restrict__ status_out) {
  for (int wi = blockIdx.x; wi < nw; wi += gridDim.x) {
    const int b = b0 + wi;
    const int count = si[(size_t)wi * kStateInts + kCount];
    for (int k = count + threadIdx.x; k < kmax; k += blockDim.x) {
      periods_out[(size_t)b * kmax + k] = 0u;
      powers_out[(size_t)b * kmax + k] = 0.0;
    }
    if (threadIdx.x == 0) {
      count_out[b] = count;
      status_out[b] = count > kmax ? PP_STATUS_OVERFLOW : PP_STATUS_OK;
    }
  }
}

// ------------------------------------------------------------------------------------------
// best-correlation
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) long_bcorr_init_kernel(LongWs w, int nw) {
  for (int wi = blockIdx.x; wi < nw; wi += gridDim.x) {
    int* si = w.si + (size_t)wi * kStateInts;
    double* sd = w.sd + (size_t)wi * kStateDbls;
    if (threadIdx.x < kStateInts) si[threadIdx.x] = threadIdx.x == kActive ? 1 : 0;
    if (threadIdx.x == 0) {
      sd[kOg] = sd[kDataNorm];
      sd[kPrev] = sd[kDataNorm];
    }
  }
}

// one round of Periods.py:321-347 per window: exact MAXABS arg-max, projection, residual, norm-drop test
__global__ void __launch_bounds__(kThreads) long_bcorr_step_kernel(LongWs w, int N, int num, int max_length, double ratio,
                                                                   int trunc_i, int orth_i, const int32_t* chain_off,
                                                                   const int32_t* chain_q, int round, int b0,
                                                                   uint32_t* __restrict__ periods_out,
                                                                   double* __restrict__ powers_out,
                                                                   double* __restrict__ bases_out) {
  __shared__ StepShared sh;
  const bool trunc = trunc_i != 0, orth = orth_i != 0;
  const double sqrtN = sqrt((double)N);
  double* v = w.vu + (size_t)blockIdx.x * 2 * w.pv;
  double* u = v + w.pv;
  const int nact = *w.count;
  for (int i = blockIdx.x; i < nact; i += gridDim.x) {
    const int wi = w.list[i];
    const int b = b0 + wi;
    int* si = w.si + (size_t)wi * kStateInts;
    double* sd = w.sd + (size_t)wi * kStateDbls;
    double* xs = w.res + (size_t)wi * w.ldr;
    const Best top = cta_argmax(w.keys + (size_t)wi * w.kld, 2, max_length - 1, PP_METRIC_MAXABS, nullptr, sh);
    uint32_t out_p = 0u;
    double out_v = 0.0;
    bool keep = false;
    if (top.p == 0) {
      if (threadIdx.x == 0) {
        si[kStatus] = PP_STATUS_NO_PERIOD;
        si[kActive] = 0;
      }
    } else {
      const int clen = orth ? chain_off[top.p + 1] - chain_off[top.p] : 0;
      cta_project_exact<false>(xs, 0, N, top.p, trunc, orth ? chain_q + chain_off[top.p] : nullptr, clen, v, u);
      cta_subtract_tiled(xs, N, v, top.p);  // always (:340)
      __syncthreads();
      const double e_now = cta_sum_sq(xs, N, sh.red);
      const double now = sqrt(e_now) / sqrtN;
      const double drop = (sd[kPrev] - now) / sd[kOg];
      if (drop > ratio) {
        keep = true;
        out_p = (uint32_t)top.p;
        out_v = drop;
      }
      __syncthreads();
      if (threadIdx.x == 0 && keep) sd[kPrev] = now;
    }
    if (threadIdx.x == 0) {
      periods_out[(size_t)b * num + round] = out_p;
      powers_out[(size_t)b * num + round] = out_v;
    }
    if (bases_out) {
      double* dst = bases_out + ((size_t)b * num + round) * N;
      if (keep) cta_store_tiled(dst, N, v, top.p);
      else
        for (int n = threadIdx.x; n < N; n += kThreads) __stcs(dst + n, 0.0);
    }
    __syncthreads();
  }
}

// rounds a window no longer takes part in (no period found): zero rows, like the on-chip kernel
__global__ void long_bcorr_final_kernel(const int* __restrict__ si, int nw, int N, int num, int b0,
                                        uint32_t* __restrict__ periods_out, double* __restrict__ powers_out,
                                        double* __restrict__ bases_out, int32_t* __restrict__ status_out) {
  for (int wi = blockIdx.x; wi < nw; wi += gridDim.x) {
    const int b = b0 + wi;
    const int status = si[(size_t)wi * kStateInts + kStatus];
    if (threadIdx.x == 0) status_out[b] = status;
    if (status == PP_STATUS_OK) continue;
    // the round that found no period wrote its own zero row; later rounds were never run for this window
    const int from = si[(size_t)wi * kStateInts + kCount];
    for (int k = from; k < num; ++k) {
      if (threadIdx.x == 0) {
        periods_out[(size_t)b * num + k] = 0u;
        powers_out[(size_t)b * num + k] = 0.0;
      }
      if (bases_out)
        for (int n = threadIdx.x; n < N; n += blockDim.x) bases_out[((size_t)b * num + k) * N + n] = 0.0;
    }
  }
}

__global__ void long_bcorr_mark_kernel(const int* __restrict__ list, const int* __restrict__ count, int* __restrict__ si,
                                       int round) {
  const int nact = *count;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nact; i += gridDim.x * blockDim.x)
    si[(size_t)list[i] * kStateInts + kCount] = round + 1;   // rounds run for this window
}

// ------------------------------------------------------------------------------------------
// best_frequency: one round, projection straight from the residual in global memory
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) long_bfreq_round_kernel(
    double* __restrict__ work, int B, int N, const double* __restrict__ mags, int F, int win, int trunc, int orth,
    const int32_t* __restrict__ chain_off, const int32_t* __restrict__ chain_q, int table_pmax,
    uint32_t* __restrict__ periods, double* __restrict__ norms, double* __restrict__ bases, int round, int num,
    int32_t* __restrict__ status, double* __restrict__ vu, int pv) {
  __shared__ double red[kWarps];
  __shared__ int redi[kWarps];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  double* v = vu + (size_t)blockIdx.x * 2 * pv;
  double* utmp = v + pv;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    if (status[b] != PP_STATUS_OK) continue;
    // np.argmax(mags): first index of the maximum; a NaN anywhere wins at its first position
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
    for (int q = 1; q < kWarps; ++q) {
      const double ob = red[q];
      const int oa = redi[q];
      const bool on = ob != ob, bn = best != best;
      const bool take = on ? (!bn || oa < arg) : (!bn && (ob > best || (ob == best && oa < arg)));
      if (take) {
        best = ob;
        arg = oa;
      }
    }
    __syncthreads();
    if (arg <= 0 || arg >= F) {
      if (tid == 0) status[b] = PP_STATUS_NO_PERIOD;
      continue;
    }
    const int p = (int)rint((2.0 * (double)win) / (double)arg);
    double* wrow = work + (size_t)b * N;
    double* brow = bases ? bases + ((size_t)b * num + round) * N : nullptr;
    double e = 0.0;
    if (p > N) {
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
      cta_project_exact<false>(wrow, 0, N, p, trunc != 0, chain, clen, v, utmp);
      const int M = N / p, r0 = N - M * p;
      for (int r = tid; r < p; r += kThreads) e = fma((double)(M + (r < r0 ? 1 : 0)) * v[r], v[r], e);
      if (brow) cta_store_tiled(brow, N, v, p);
      cta_subtract_tiled(wrow, N, v, p);
    }
    e = warp_sum(e);
    __syncthreads();
    if (lane == 0) red[wid] = e;
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
      for (int q = 0; q < kWarps; ++q) t += red[q];
      periods[(size_t)b * num + round] = (uint32_t)p;
      norms[(size_t)b * num + round] = sqrt(t) / sqrt((double)N);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int carve_long(int algo, int B, int N, int pmax, int num, int orth, const DeviceFacts& f, void* ws, size_t bytes,
                      LongWs& w) {
  const size_t need = long_layout(algo, B, N, pmax, num, orth, f, ws, bytes, w);
  if (ws == nullptr || bytes < need) return fail(-3, "workspace too small (see pp_long_workspace_bytes)%s");
  return 0;
}

}  // namespace
}  // namespace pp

using namespace pp;

extern "C" {

size_t pp_long_workspace_bytes(int32_t algo, int32_t B, int32_t N, int32_t pmax, int32_t num, int32_t orth) {
  if (B < 1 || N < 2 || pmax < 1 || num < 0) return 0;
  if (algo != PP_ALGO_PROJECT && algo != PP_ALGO_SWEEP && algo != PP_ALGO_MBEST && algo != PP_ALGO_S2L &&
      algo != PP_ALGO_BCORR && algo != PP_ALGO_BFREQ)
    return 0;
  DeviceFacts f;
  if (device_facts(f)) return 0;
  LongWs w;
  return long_layout(algo, B, N, pmax, num, orth, f, nullptr, 0, w);
}

int pp_long_project(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t p, int32_t trunc,
                    const int32_t* chain_q_host, int32_t chain_len, double* out, int64_t ldo, int32_t out_len,
                    void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;
  if (int rc = check_common_long(x, ldx, B, N)) return rc;
  if (p < 1 || p > N) return fail(-1, "period must satisfy 1 <= p <= N%s");
  if (chain_len < 0 || chain_len > 16) return fail(-1, "chain_len must be in [0,16]%s");
  if (out == nullptr || out_len < 1 || out_len > N || ldo < out_len) return fail(-1, "bad output shape%s");
  ChainArgL ca;
  memset(&ca, 0, sizeof(ca));
  ca.len = chain_len;
  for (int i = 0; i < chain_len; ++i) {
    if (chain_q_host[i] < 1 || chain_q_host[i] >= p || p % chain_q_host[i]) return fail(-1, "chain cofactor must divide p%s");
    ca.q[i] = chain_q_host[i];
  }
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  LongWs w;
  if (int rc = carve_long(PP_ALGO_PROJECT, B, N, p, 0, 0, f, workspace, workspace_bytes, w)) return rc;
  long_project_kernel<<<w.grid, kThreads, 0, (cudaStream_t)stream>>>(x, ldx, B, N, p, trunc, ca, out, ldo, out_len, w.vu,
                                                                     w.pv);
  return check_cuda(cudaGetLastError(), "long_project_kernel launch");
}

int pp_long_sweep(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t pmin, int32_t pmax, int32_t metric,
                  int32_t trunc, int32_t orth, const int32_t* chain_off, const int32_t* chain_q, int32_t table_pmax,
                  double* metric_out, int32_t* best_p, double* best_val, void* workspace, size_t workspace_bytes,
                  void* stream) {
  if (B == 0) return 0;
  if (int rc = check_common_long(x, ldx, B, N)) return rc;
  if (pmin < 1 || pmax < pmin || pmax > N) return fail(-1, "need 1 <= pmin <= pmax <= N%s");
  if (metric < 0 || metric > 3) return fail(-1, "unknown metric%s");
  if (metric == PP_METRIC_MAXABS && (trunc || orth)) return fail(-1, "MAXABS ignores trunc/orth; pass 0%s");
  if (orth && (chain_off == nullptr || chain_q == nullptr || table_pmax < pmax)) return fail(-1, "orth needs tables covering pmax%s");
  if (best_p == nullptr || best_val == nullptr) return fail(-1, "best_p/best_val are null%s");
  cudaStream_t s = (cudaStream_t)stream;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  LongWs w;
  if (int rc = carve_long(PP_ALGO_SWEEP, B, N, pmax, 0, orth, f, workspace, workspace_bytes, w)) return rc;
  for (int b0 = 0; b0 < B; b0 += w.piece) {
    const int nw = B - b0 < w.piece ? B - b0 : w.piece;
    long_load_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(x + (size_t)b0 * ldx, ldx, nw, N, w.res, w.ldr, w.sd);
    long_activate_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(w, nw);
    int nact = 0;
    if (int rc = active_windows(w, nw, s, nact)) return rc;
    if (int rc = launch_sweep(w, N, pmin, pmax, pmax - pmin + 1, false, metric, trunc, orth, chain_off, chain_q, f, s))
      return rc;
    long_sweep_step_kernel<<<step_grid(w, nact), kThreads, 0, s>>>(w, N, pmin, pmax, metric, trunc, orth, chain_off,
                                                                   chain_q, metric_out, best_p, best_val, b0);
    if (int rc = check_cuda(cudaGetLastError(), "long_sweep_step_kernel launch")) return rc;
  }
  return 0;
}

int pp_long_mbest(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t num, int32_t pmin, int32_t pmax,
                  int32_t gamma, int32_t trunc, int32_t orth, const int32_t* chain_off, const int32_t* chain_q,
                  const int32_t* fac_off, const int32_t* fac, int32_t table_pmax, uint32_t* periods, double* powers,
                  double* bases, int32_t* sweeps, int32_t* near_ties, int32_t* status, void* workspace,
                  size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;
  if (int rc = check_common_long(x, ldx, B, N)) return rc;
  if (num < 1 || num > 4096) return fail(-1, "need 1 <= num <= 4096%s");
  if (pmin < 2 || pmax < pmin || pmax > N) return fail(-1, "need 2 <= pmin <= pmax <= N%s");
  if (pmax - pmin + 1 < num) return fail(-1, "fewer candidate periods than num%s");
  if (fac_off == nullptr || fac == nullptr || table_pmax < pmax) return fail(-1, "factor tables must cover pmax%s");
  if (orth && (chain_off == nullptr || chain_q == nullptr)) return fail(-1, "orth needs chain tables%s");
  if (!periods || !powers || !status) return fail(-1, "output pointers are null%s");
  cudaStream_t s = (cudaStream_t)stream;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  LongWs w;
  if (int rc = carve_long(PP_ALGO_MBEST, B, N, pmax, num, orth, f, workspace, workspace_bytes, w)) return rc;
  const int metric = gamma ? PP_METRIC_GAMMA : PP_METRIC_NORM;
  const int guard = 12 * (pmax - pmin + 2) + 12 * num;
  for (int b0 = 0; b0 < B; b0 += w.piece) {
    const int nw = B - b0 < w.piece ? B - b0 : w.piece;
    long_load_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(x + (size_t)b0 * ldx, ldx, nw, N, w.res, w.ldr, w.sd);
    long_mbest_init_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(w, nw, num);
    while (true) {
      int nact = 0;
      if (int rc = active_windows(w, nw, s, nact)) return rc;
      if (nact == 0) break;
      if (int rc = launch_sweep(w, N, pmin, pmax, pmax - pmin + 1, false, metric, trunc, orth, chain_off, chain_q, f, s))
        return rc;
      long_mbest_step_kernel<<<step_grid(w, nact), kThreads, 0, s>>>(w, N, num, pmin, pmax, gamma, trunc, orth,
                                                                     chain_off, chain_q, guard);
      if (int rc = check_cuda(cudaGetLastError(), "long_mbest_step_kernel launch")) return rc;
    }
    long_mbest_final_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(w, nw, N, num, pmax, gamma, trunc, orth, chain_off,
                                                                  chain_q, fac_off, fac, b0, periods, powers, bases,
                                                                  sweeps, near_ties, status);
    if (int rc = check_cuda(cudaGetLastError(), "long_mbest_final_kernel launch")) return rc;
  }
  return 0;
}

int pp_long_small_to_large(const double* x, int64_t ldx, int32_t B, int32_t N, double thresh, int32_t n_periods,
                           int32_t trunc, int32_t orth, const int32_t* chain_off, const int32_t* chain_q,
                           int32_t table_pmax, int32_t kmax, uint32_t* periods, double* powers, double* bases,
                           int32_t* count, int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;
  if (int rc = check_common_long(x, ldx, B, N)) return rc;
  if (!(thresh >= 0.0)) return fail(-1, "thresh must be >= 0%s");
  if (n_periods < 2 || n_periods > N) return fail(-1, "need 2 <= n_periods <= N%s");
  if (kmax < 1) return fail(-1, "kmax must be >= 1%s");
  if (orth && (chain_off == nullptr || chain_q == nullptr || table_pmax < n_periods)) return fail(-1, "orth needs tables covering n_periods%s");
  if (!periods || !powers || !count || !status) return fail(-1, "output pointers are null%s");
  cudaStream_t s = (cudaStream_t)stream;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  LongWs w;
  if (int rc = carve_long(PP_ALGO_S2L, B, N, n_periods, 0, orth, f, workspace, workspace_bytes, w)) return rc;
  for (int b0 = 0; b0 < B; b0 += w.piece) {
    const int nw = B - b0 < w.piece ? B - b0 : w.piece;
    long_load_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(x + (size_t)b0 * ldx, ldx, nw, N, w.res, w.ldr, w.sd);
    long_activate_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(w, nw);
    while (true) {
      int nact = 0;
      if (int rc = active_windows(w, nw, s, nact)) return rc;
      if (nact == 0) break;
      // candidates per window and round: enough units for every warp of the grid; the speculation past a hit is
      // bounded by this chunk (the result does not depend on it)
      int span = (w.grid * kWarps + nact - 1) / nact;
      span = span < kS2lMinChunk ? kS2lMinChunk : (span > kS2lMaxChunk ? kS2lMaxChunk : span);
      if (int rc = launch_sweep(w, N, 2, n_periods, span, true, PP_METRIC_IMPOSED, trunc, orth, chain_off, chain_q, f, s))
        return rc;
      long_s2l_step_kernel<<<step_grid(w, nact), kThreads, 0, s>>>(w, N, thresh, n_periods, span, trunc, orth, chain_off,
                                                                   chain_q, kmax, b0, periods, powers, bases);
      if (int rc = check_cuda(cudaGetLastError(), "long_s2l_step_kernel launch")) return rc;
    }
    long_s2l_final_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(w.si, nw, kmax, b0, periods, powers, count, status);
    if (int rc = check_cuda(cudaGetLastError(), "long_s2l_final_kernel launch")) return rc;
  }
  return 0;
}

int pp_long_best_correlation(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t num, int32_t max_length,
                             double ratio, int32_t trunc, int32_t orth, const int32_t* chain_off, const int32_t* chain_q,
                             int32_t table_pmax, uint32_t* periods, double* powers, double* bases, int32_t* status,
                             void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;
  if (int rc = check_common_long(x, ldx, B, N)) return rc;
  if (num < 1) return fail(-1, "num must be >= 1%s");
  if (max_length < 3 || max_length > N + 1) return fail(-1, "need 3 <= max_length <= N+1%s");
  if (orth && (chain_off == nullptr || chain_q == nullptr || table_pmax < max_length - 1)) return fail(-1, "orth needs tables covering max_length%s");
  if (!periods || !powers || !status) return fail(-1, "output pointers are null%s");
  cudaStream_t s = (cudaStream_t)stream;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  LongWs w;
  if (int rc = carve_long(PP_ALGO_BCORR, B, N, max_length, 0, orth, f, workspace, workspace_bytes, w)) return rc;
  for (int b0 = 0; b0 < B; b0 += w.piece) {
    const int nw = B - b0 < w.piece ? B - b0 : w.piece;
    long_load_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(x + (size_t)b0 * ldx, ldx, nw, N, w.res, w.ldr, w.sd);
    long_bcorr_init_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(w, nw);
    for (int round = 0; round < num; ++round) {
      int nact = 0;
      if (int rc = active_windows(w, nw, s, nact)) return rc;
      if (nact == 0) break;
      // the correlation metric always folds all N samples (trunc / orth only shape the projection)
      if (int rc = launch_sweep(w, N, 2, max_length - 1, max_length - 2, false, PP_METRIC_MAXABS, 0, 0, nullptr, nullptr,
                                f, s))
        return rc;
      long_bcorr_mark_kernel<<<1, kThreads, 0, s>>>(w.list, w.count, w.si, round);
      long_bcorr_step_kernel<<<step_grid(w, nact), kThreads, 0, s>>>(w, N, num, max_length, ratio, trunc, orth,
                                                                     chain_off, chain_q, round, b0, periods, powers,
                                                                     bases);
      if (int rc = check_cuda(cudaGetLastError(), "long_bcorr_step_kernel launch")) return rc;
    }
    long_bcorr_final_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(w.si, nw, N, num, b0, periods, powers, bases, status);
    if (int rc = check_cuda(cudaGetLastError(), "long_bcorr_final_kernel launch")) return rc;
  }
  return 0;
}

int pp_long_best_frequency_round(double* work, int32_t B, int32_t N, const double* mags, int32_t F, int32_t win_size,
                                 int32_t trunc, int32_t orth, const int32_t* chain_off, const int32_t* chain_q,
                                 int32_t table_pmax, uint32_t* periods, double* norms, double* bases, int32_t round,
                                 int32_t num, int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;
  if (!work || !mags || !periods || !norms || !status || B < 0 || N < 2 || F < 2 || win_size < 2 || num < 1 || round < 0 ||
      round >= num)
    return fail(-1, "bad best_frequency arguments%s");
  if (orth && (!chain_off || !chain_q)) return fail(-1, "orthogonalize needs the cofactor-chain tables%s");
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  LongWs w;
  if (int rc = carve_long(PP_ALGO_BFREQ, B, N, N, 0, 0, f, workspace, workspace_bytes, w)) return rc;
  long_bfreq_round_kernel<<<step_grid(w, B), kThreads, 0, (cudaStream_t)stream>>>(
      work, B, N, mags, F, win_size, trunc, orth, chain_off, chain_q, table_pmax, periods, norms, bases, round, num, status,
      w.vu, w.pv);
  return check_cuda(cudaGetLastError(), "long_bfreq_round_kernel launch");
}

}  // extern "C"
