// pyperiod_b200 -- the global-memory ("long") path of QOPeriods and of the Muresan finder: windows whose on-chip
// plan does not fit the shared memory of one CTA (pp_qo_fits_on_chip).  Same results contract as qo_find_kernel,
// qo_solve_kernel and muresan_kernel, which stay untouched.
//
// Layout.  Batches run in pieces of windows.  Each window of a piece owns, in the workspace: its residual row (zero
// padded, as pp_long.cu), its integer state (found periods, dictionary, divisor bitmap -- the QoCtx block the
// on-chip kernels keep in shared memory), its packed Cholesky factor (natural basis) or conjugate-gradient vectors
// (Ramanujan basis), the weights saved by the refinement step and its round norms.  The factor survives from round
// to round, so the incremental factorisation (row_lo) works as on chip.  The piece is the smaller of half the L2
// cache in residuals and what the workspace holds in factors.
//
// find_periods rounds, driven by the host on the caller's stream:
//   sweep   long_sweep_kernel, PP_METRIC_GAMMA, no orthogonalisation: energies of the on-chip direct fold.
//   step    one CTA per active window: arg-max with the rule of cta_sweep (E/p by cross multiplication, strict '>',
//           lowest p on ties; no near-tie audit, as qo_find_kernel runs none), then cta_qo_solve / cta_qo_solve_ram
//           unchanged on a QoCtx whose window (x0, read in place), residual, factor and integer state are in global
//           memory.  Only the right-hand side / weights (wv) and the factorisation's staging area are in shared
//           memory; wv bounds the dictionary (pp_long_qo_max_rows).  Then qo_commit and the reference's stop test.
//   The host reads the number of windows still active (4 bytes) once per round and stops at 0.
// The solve stage alone (either basis) is one step per window.  Muresan: one warp per (window, q) folds from global
// memory with muresan_kernel's lane-to-residue mapping and summation order, then one CTA per window runs the Moebius
// pass.
//
// Index widths: packed-factor offsets are size_t (pp_chol.cuh), row and sample indices stay below N < 2^31.  The
// 32767 cap of the on-chip launches comes from the hierarchical fold's 16-bit job descriptors; this path folds
// directly and has no such cap.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pyperiod_b200.h"
#include "pp_common.cuh"
#include "pp_sweep.cuh"
#include "pp_chol.cuh"
#include "pp_host.cuh"
#include "pp_long.cuh"
#include "pp_qo.cuh"

namespace pp {
namespace {

// shared memory of a step CTA: factorisation staging (Bs, then D / Li / rD / flag), wv, the reduction scratch
constexpr size_t kStepChol = (kCholStageD + 15) & ~(size_t)15;
__host__ __device__ inline size_t long_qo_smem(int wv_len) {
  return kCholStageBs + kStepChol + (size_t)wv_len * 8 + 2 * kWarps * 8;
}

// rows of the largest dictionary a step CTA holds with smem_bytes of shared memory (wv = rows + 2 kCb doubles)
inline int long_qo_rows(size_t smem_bytes) {
  const size_t fixed = long_qo_smem(2 * kCb) + sizeof(StepShared) + 1024;
  if (smem_bytes <= fixed) return 0;
  return (int)(((smem_bytes - fixed) / 8) / kCb * kCb);
}

struct LongQo {
  LongWs w;                 // res, keys, sd, si, list, count, counter of the round loop
  QoPlan pl;                // per-window sizes: rmax, wv_len, seen_words, ws_L, cg_len
  int ints = 0;             // ints of per-window state (the QoCtx block of make_ctx)
  size_t l_len = 0;         // doubles of factor / conjugate-gradient vectors per window
  int u_len = 0;            // doubles of A^T p per window (Ramanujan basis)
  int* ctx = nullptr;       // [piece, ints]
  double* L = nullptr;      // [piece, l_len]
  double* wsave = nullptr;  // [piece, wv_len]
  double* u = nullptr;      // [piece, u_len]
  double* rnorms = nullptr; // [piece, num]
};

// Sizes (base == nullptr) or carves the workspace for `piece` windows.  Returns the bytes needed.
size_t long_qo_carve(bool find, int piece, int N, int pmax, int num, int rmax, bool ram, int grid, void* base,
                     size_t bytes, LongQo& q) {
  q.pl = make_qo_plan(N, pmax, num, rmax, false, ram, true);
  q.ints = 8 * num + 2 + q.pl.seen_words + 16;
  q.l_len = q.pl.ws_L() / 8;
  q.u_len = ram ? q.pl.u_len : 0;
  LongWs& w = q.w;
  w.ldr = long_ldr(N);
  w.kld = pmax + 1;
  w.pv = 0;
  w.num = num;
  w.piece = piece;
  w.grid = grid;
  size_t off = 0;
  auto take = [&](size_t n) -> void* {
    off = (off + 255) & ~(size_t)255;
    void* p = (base != nullptr && off + n <= bytes) ? (void*)((char*)base + off) : nullptr;
    off += n;
    return p;
  };
  const size_t P = (size_t)piece;
  w.res = (double*)take(P * w.ldr * 8);
  q.ctx = (int*)take(P * q.ints * 4);
  q.L = (double*)take(P * q.l_len * 8);
  q.wsave = (double*)take(P * q.pl.wv_len() * 8);
  q.u = ram ? (double*)take(P * q.u_len * 8) : nullptr;
  if (find) {
    w.keys = (double*)take(P * w.kld * 8);
    w.sd = (double*)take(P * kStateDbls * 8);
    w.si = (int*)take(P * kStateInts * 4);
    w.list = (int*)take(P * 4);
    w.count = (int*)take(256);
    w.counter = (int*)take(256);
    q.rnorms = (double*)take(P * num * 8);
  }
  return off + 256;
}

// windows per piece: half the L2 cache in residuals, at most B, and what `bytes` holds
int long_qo_piece(bool find, int B, int N, int pmax, int num, int rmax, bool ram, size_t bytes) {
  LongQo q;
  size_t piece = (size_t)l2_bytes() / 2 / ((size_t)long_ldr(N) * 8);
  if (piece < 1) piece = 1;
  if (piece > (size_t)B) piece = (size_t)B;
  const size_t one = long_qo_carve(find, 1, N, pmax, num, rmax, ram, 0, nullptr, 0, q);
  const size_t per = long_qo_carve(find, 2, N, pmax, num, rmax, ram, 0, nullptr, 0, q) - one;
  if (bytes < one) return 0;
  const size_t fit = 1 + (bytes - one) / (per + 2048);   // 2048: the 256-byte alignment of each array
  return (int)(piece < fit ? piece : fit);
}

struct LongQoArgs {
  const double* x;
  int64_t ldx;
  const int32_t* order;   // window of slot i of the launch: order[i], or i (nullable)
  int b0;                 // first slot of the piece
  int N, num, pmin, pmax, trunc, refine, rmax, wv_len, u_len, cg_len, seen_words, ints;
  size_t l_len;
  double thresh;
  const int32_t* phi;
  int* ctx;
  double* L;
  double* wsave;
  double* u;
  double* rnorms;
  LongWs w;
  __device__ int window(int wi) const { return order ? order[b0 + wi] : b0 + wi; }
};

// QoCtx of window wi of the piece: integer state, residual, factor in global memory; wv and staging in shared
__device__ QoCtx long_qo_ctx(const LongQoArgs& a, int wi, const double* x0, long long* timers) {
  unsigned char* smem = pp_smem;
  QoCtx c;
  c.N = a.N;
  c.num = a.num;
  c.rmax = a.rmax;
  c.refine = a.refine;
  c.phi = a.phi;
  c.x0 = x0;
  c.xs = a.w.res + (size_t)wi * a.w.ldr;
  c.cs.Bs = reinterpret_cast<double*>(smem);
  double* chol = reinterpret_cast<double*>(smem + kCholStageBs);
  c.cs.D = chol;
  c.cs.Li = chol + kCb * kLdD;
  c.cs.rD = c.cs.Li + kCb * kLdD;
  c.cs.flag = reinterpret_cast<int*>(c.cs.rD + kCb);
  c.wv = reinterpret_cast<double*>(smem + kCholStageBs + kStepChol);
  c.red = c.wv + a.wv_len;
  int* ints = a.ctx + (size_t)wi * a.ints;
  c.found = ints;
  c.dict_q = ints + a.num;
  c.dict_keep = ints + 2 * a.num;
  c.dict_rows = ints + 3 * a.num;
  c.dict_off = ints + 4 * a.num;
  c.prev_rows = ints + 5 * a.num + 1;
  c.seen = reinterpret_cast<uint32_t*>(ints + 7 * a.num + 1);
  c.seen_words = a.seen_words;
  c.misc = ints + 7 * a.num + 1 + a.seen_words;
  c.tab_off = c.misc + 16;
  c.L = a.L + (size_t)wi * a.l_len;
  c.wsave = a.wsave + (size_t)wi * a.wv_len;
  c.u = a.u ? a.u + (size_t)wi * a.u_len : nullptr;
  c.cg_len = a.cg_len;
  c.t = timers;
  return c;
}

// round 0 of every window of the piece: the outputs of a window nothing could be solved for, the zero-signal early
// out (QOPeriods.py:394-406), the state of the round loop.  Residual rows and sd[kEres] come from long_load_kernel.
__global__ void __launch_bounds__(kThreads) long_qo_init_kernel(LongQoArgs a, QoOut out, int nw) {
  const int tid = threadIdx.x;
  __shared__ double red[kWarps];
  for (int wi = blockIdx.x; wi < nw; wi += gridDim.x) {
    const int b = a.window(wi);
    const double* x0 = a.x + (size_t)b * a.ldx;
    QoCtx c = long_qo_ctx(a, wi, x0, nullptr);
    double sa = 0.0;
    for (int n = tid; n < a.N; n += kThreads) sa += fabs(x0[n]);
    sa = warp_sum(sa);
    if ((tid & 31) == 0) red[tid >> 5] = sa;
    __syncthreads();
    double sum_abs = 0.0;
    for (int w = 0; w < kWarps; ++w) sum_abs += red[w];
    if (tid == 0) {
      c.misc[0] = 0;
      c.misc[1] = 0;
      c.misc[8] = 0;
      c.misc[9] = 0;
      c.misc[11] = -1;
    }
    __syncthreads();
    qo_commit(c, out, b, 0, a.rnorms + (size_t)wi * a.num);
    const bool zero = sum_abs <= 1e-16;
    if (zero && out.res)
      for (int n = tid; n < a.N; n += kThreads) out.res[(size_t)b * a.N + n] = 0.0;
    if (tid == 0) {
      int* si = a.w.si + (size_t)wi * kStateInts;
      for (int k = 0; k < kStateInts; ++k) si[k] = 0;
      si[kActive] = zero ? 0 : 1;
      out.status[b] = zero ? PP_STATUS_ZERO_INPUT : PP_STATUS_OK;
    }
    __syncthreads();
  }
}

// one round of QOPeriods.py:417-594 for every active window: arg-max of the sweep, solve, commit, stop test
template <int BASIS>
__global__ void __launch_bounds__(kThreads) long_qo_step_kernel(LongQoArgs a, QoOut out, int round) {
  __shared__ StepShared sh;
  const int tid = threadIdx.x;
  const double sqrtN = sqrt((double)a.N);
  long long timers[6] = {0, 0, 0, 0, 0, 0};
  const int nact = *a.w.count;
  for (int i = blockIdx.x; i < nact; i += gridDim.x) {
    const int wi = a.w.list[i];
    const int b = a.window(wi);
    QoCtx c = long_qo_ctx(a, wi, a.x + (size_t)b * a.ldx, timers);
    int* si = a.w.si + (size_t)wi * kStateInts;
    double* sd = a.w.sd + (size_t)wi * kStateDbls;
    double* rnorms = a.rnorms + (size_t)wi * a.num;
    const Best top = cta_argmax(a.w.keys + (size_t)wi * a.w.kld, a.pmin, a.pmax, PP_METRIC_GAMMA, nullptr, sh);
    int nfound = si[kFilled];
    __syncthreads();
    if (tid == 0) {
      rnorms[round] = top.p != 0 ? key_to_value(PP_METRIC_GAMMA, top.key, top.p, sqrtN) : 0.0;
      if (top.p > 0) c.found[nfound] = top.p;
    }
    if (top.p > 0) ++nfound;
    __syncthreads();
    double e_recon = 0.0;
    const int rc = BASIS == 1 ? cta_qo_solve_ram(c, nfound, &e_recon) : cta_qo_solve(c, nfound, &e_recon);
    if (rc != PP_STATUS_OK) {   // LinAlgError in the reference: keep the previous round's outputs (:552-559)
      if (tid == 0) {
        out.status[b] = rc;
        if (rc == PP_STATUS_TOO_LARGE) out.n_weights[b] = c.misc[1];   // the rows a re-run needs
        si[kActive] = 0;
      }
      __syncthreads();
      continue;
    }
    qo_commit(c, out, b, nfound, rnorms);
    // default test_function: rms(reconstruction) > rms(data) * thresh (QOPeriods.py:391), ahead of the next round
    const bool last = round + 1 >= a.num;
    const bool go = !last && sqrt(e_recon / (double)a.N) > sqrt(sd[kEres] / (double)a.N) * a.thresh;
    __syncthreads();
    if (tid == 0) {
      si[kFilled] = nfound;
      if (!go) {
        // a stop keeps the weights of all periods but does not report the last one (QOPeriods.py:560-594)
        out.n_periods[b] = last ? nfound : (nfound > 0 ? nfound - 1 : 0);
        si[kActive] = 0;
      }
    }
    __syncthreads();
  }
}

// solve stage alone (qo_solve_kernel with the window in place and the factor -- or, for the Ramanujan basis, the
// conjugate-gradient vectors -- per window)
template <int BASIS>
__global__ void __launch_bounds__(kThreads) long_qo_solve_kernel(LongQoArgs a, int nw, const int32_t* __restrict__ entries,
                                                                 const int32_t* __restrict__ explicit_rows,
                                                                 const int32_t* __restrict__ n_entries, int kmax,
                                                                 QoOut out) {
  const int tid = threadIdx.x;
  long long timers[6] = {0, 0, 0, 0, 0, 0};
  for (int wi = blockIdx.x; wi < nw; wi += gridDim.x) {
    const int b = a.window(wi);
    const double* x0 = a.x + (size_t)b * a.ldx;
    QoCtx c = long_qo_ctx(a, wi, x0, timers);
    const int nd = min(max(n_entries[b], 0), kmax);
    if (explicit_rows == nullptr) {
      for (int i = tid; i < nd; i += kThreads) c.found[i] = entries[(size_t)b * kmax + i];
      if (tid == 0) c.misc[8] = c.misc[9] = 0;
    } else if (tid == 0) {
      int off = 0;
      for (int k = 0; k < nd; ++k) {
        const int q = entries[(size_t)b * kmax + k];
        int rows = explicit_rows[(size_t)b * kmax + k];
        rows = rows > 0 && rows <= q ? rows : q;   // 0 keeps every row (QOPeriods.py:972)
        c.dict_q[k] = q;
        c.dict_keep[k] = rows;
        c.dict_rows[k] = rows;
        c.dict_off[k] = off;
        off += rows;
      }
      c.dict_off[nd] = off;
      c.misc[0] = nd;
      c.misc[1] = off;
      c.misc[8] = c.misc[9] = 0;
    }
    __syncthreads();
    double e_recon = 0.0;
    const int rc = BASIS == 1 ? cta_qo_solve_ram(c, nd, &e_recon) : cta_qo_solve(c, nd, &e_recon, explicit_rows != nullptr);
    const int ndict = c.misc[0], R = c.misc[1];
    if (rc == PP_STATUS_OK) {
      if (out.dict_q != nullptr)
        for (int i = tid; i < kmax; i += kThreads) {
          out.dict_q[(size_t)b * kmax + i] = i < ndict ? c.dict_q[i] : 0;
          out.dict_keep[(size_t)b * kmax + i] = i < ndict ? c.dict_keep[i] : 0;
        }
      double* w = out.weights_of(b);
      for (int i = tid; i < R; i += kThreads) w[i] = c.wv[i];
      if (out.res)
        for (int n = tid; n < a.N; n += kThreads) out.res[(size_t)b * a.N + n] = c.xs[n];
    } else if (out.res) {
      for (int n = tid; n < a.N; n += kThreads) out.res[(size_t)b * a.N + n] = x0[n];
    }
    if (tid == 0) {
      if (out.n_dict != nullptr) out.n_dict[b] = rc == PP_STATUS_OK ? ndict : 0;
      out.n_weights[b] = rc == PP_STATUS_OK ? R : (rc == PP_STATUS_TOO_LARGE ? R : 0);
      out.status[b] = rc;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// Muresan eq. 3
// ------------------------------------------------------------------------------------------
// raw[w, q] = max(eq_3, 0) for q in [1, max_p), one warp per (window, q): muresan_kernel's fold and lag sums on the
// window in global memory, same lanes, same order
__global__ void __launch_bounds__(kThreads) long_muresan_raw_kernel(const double* __restrict__ x, int64_t ldx, int b0,
                                                                    int nw, int N, int max_p, double* __restrict__ raw,
                                                                    double* __restrict__ raw_out) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * kWarps;
  const long long total = (long long)nw * (max_p - 1);
  for (long long u = (long long)blockIdx.x * kWarps + (threadIdx.x >> 5); u < total; u += warps) {
    const int q = 1 + (int)(u / nw);
    const int wi = (int)(u - (long long)(q - 1) * nw);
    const int b = b0 + wi;
    const double* xs = x + (size_t)b * ldx;
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
      raw[(size_t)wi * max_p + q] = fmax(v, 0.0);
      if (raw_out) raw_out[(size_t)b * max_p + q] = v;
    }
  }
}

// pows[b, q] = sum_{d | q} mu(q / d) raw[d], clamp, optional / q, first arg-max (muresan_kernel's second half)
__global__ void __launch_bounds__(kThreads) long_muresan_final_kernel(const double* __restrict__ raw, int b0, int nw,
                                                                      int max_p, int normalize,
                                                                      const int32_t* __restrict__ mu,
                                                                      double* __restrict__ raw_out,
                                                                      double* __restrict__ pows_out,
                                                                      int32_t* __restrict__ best_out) {
  __shared__ double red[kWarps];
  __shared__ int redi[kWarps];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  for (int wi = blockIdx.x; wi < nw; wi += gridDim.x) {
    const int b = b0 + wi;
    const double* rw = raw + (size_t)wi * max_p;
    if (tid == 0 && raw_out) raw_out[(size_t)b * max_p] = 0.0;
    double best = -1.0;
    int arg = 0;
    for (int q = tid; q < max_p; q += kThreads) {
      double v = 0.0;
      if (q >= 1) {
        for (int d = 1; d * d <= q; ++d) {
          if (q % d) continue;
          const int d2 = q / d;
          v += (double)mu[d2] * rw[d];
          if (d2 != d) v += (double)mu[d] * rw[d2];
        }
        if (v < 0.0) v = 0.0;
        if (normalize) v = v / (double)q;
      }
      if (pows_out) pows_out[(size_t)b * max_p + q] = v;
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
      best_out[b] = arg > 0 ? arg : 1;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
size_t muresan_piece_bytes(int max_p) { return (size_t)max_p * 8; }

int muresan_piece(int B, int max_p) {
  size_t piece = (size_t)l2_bytes() / 2 / muresan_piece_bytes(max_p);
  if (piece < 1) piece = 1;
  if (piece > (size_t)B) piece = (size_t)B;
  return (int)piece;
}

LongQoArgs long_qo_args(const LongQo& q, const double* x, int64_t ldx, const int32_t* order, int N, int num, int pmin,
                        int pmax, int trunc, int refine, double thresh, const int32_t* phi) {
  LongQoArgs a;
  a.x = x;
  a.ldx = ldx;
  a.order = order;
  a.b0 = 0;
  a.N = N;
  a.num = num;
  a.pmin = pmin;
  a.pmax = pmax;
  a.trunc = trunc;
  a.refine = refine;
  a.rmax = q.pl.rmax;
  a.wv_len = q.pl.wv_len();
  a.u_len = q.u_len;
  a.cg_len = q.pl.cg_len;
  a.seen_words = q.pl.seen_words;
  a.ints = q.ints;
  a.l_len = q.l_len;
  a.thresh = thresh;
  a.phi = phi;
  a.ctx = q.ctx;
  a.L = q.L;
  a.wsave = q.wsave;
  a.u = q.u;
  a.rnorms = q.rnorms;
  a.w = q.w;
  return a;
}

// rows of the largest dictionary on this device, and the plan rmax of a call: rmax rounded up to kCb, capped
int device_rows(const DeviceFacts& f) { return long_qo_rows((size_t)f.smem_optin); }

int prepare(const DeviceFacts& f, int rmax, bool find, int B, int N, int pmax, int num, bool ram, void* workspace,
            size_t workspace_bytes, LongQo& q, int& rmax_eff) {
  const int cap = device_rows(f);
  if (cap < kCb) return fail(-2, "not enough shared memory for the long-path step%s");
  rmax_eff = (rmax + kCb - 1) / kCb * kCb;
  if (rmax_eff > cap) rmax_eff = cap;
  const int piece = long_qo_piece(find, B, N, pmax, num, rmax_eff, ram, workspace_bytes);
  if (workspace == nullptr || piece < 1) return fail(-3, "workspace too small (see pp_long_qo_workspace_bytes)%s");
  long_qo_carve(find, piece, N, pmax, num, rmax_eff, ram, f.sm_count * kLongCtasPerSm, workspace, workspace_bytes, q);
  return 0;
}

int long_qo_solve_launch(const double* x, int64_t ldx, int B, int N, int kmax, const int32_t* entries,
                         const int32_t* explicit_rows, const int32_t* n_entries, int pmax, int refine, const int32_t* phi,
                         int rmax, const int32_t* order, int n_order, QoOut o, void* workspace, size_t workspace_bytes,
                         cudaStream_t s, bool ram = false) {
  const int count = order ? n_order : B;
  if (count == 0) return 0;
  if (count < 0 || count > B) return fail(-1, "bad order list%s");
  if (refine < 0 || refine > 4) return fail(-1, "refine must be in [0, 4]%s");
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  LongQo q;
  int rmax_eff = 0;
  if (int rc = prepare(f, rmax, false, count, N, pmax, kmax, ram, workspace, workspace_bytes, q, rmax_eff)) return rc;
  if (o.weights_off == nullptr && o.ldw < q.pl.rmax)
    return fail(-1, "ldw must be >= rmax rounded up to a multiple of 32 (or pass weights_off)%s");
  const size_t smem = long_qo_smem(q.pl.wv_len());
  if (int rc = ram ? prep_kernel(long_qo_solve_kernel<1>, smem, f) : prep_kernel(long_qo_solve_kernel<0>, smem, f))
    return rc;
  LongQoArgs a = long_qo_args(q, x, ldx, order, N, kmax, 1, pmax, 0, refine, 0.0, phi);
  for (int b0 = 0; b0 < count; b0 += q.w.piece) {
    const int nw = count - b0 < q.w.piece ? count - b0 : q.w.piece;
    a.b0 = b0;
    if (ram)
      long_qo_solve_kernel<1><<<step_grid(q.w, nw), kThreads, smem, s>>>(a, nw, entries, nullptr, n_entries, kmax, o);
    else
      long_qo_solve_kernel<0><<<step_grid(q.w, nw), kThreads, smem, s>>>(a, nw, entries, explicit_rows, n_entries, kmax,
                                                                         o);
    if (int rc = check_cuda(cudaGetLastError(), "long_qo_solve_kernel launch")) return rc;
  }
  return check_cuda(cudaStreamSynchronize(s), "cudaStreamSynchronize");
}

int check_qo_long(const void* x, int64_t ldx, int B, int N, int num, int pmax, int rmax, const void* phi, int table_pmax) {
  if (int rc = check_common_long(x, ldx, B, N)) return rc;
  if (num < 1 || num > 256) return fail(-1, "need 1 <= num <= 256%s");
  if (pmax < 1 || pmax > N) return fail(-1, "need 1 <= pmax <= N%s");
  if (rmax < 2) return fail(-1, "rmax must be >= 2%s");
  if (table_pmax >= 0 && (phi == nullptr || table_pmax < pmax)) return fail(-1, "phi table must cover pmax%s");
  return 0;
}

}  // namespace
}  // namespace pp

using namespace pp;

extern "C" {

int32_t pp_long_qo_max_rows(int32_t smem_bytes) { return smem_bytes < 0 ? 0 : long_qo_rows((size_t)smem_bytes); }

size_t pp_long_qo_workspace_bytes(int32_t kind, int32_t B, int32_t N, int32_t pmax, int32_t num, int32_t rmax,
                                  int32_t basis, size_t factor_budget) {
  if (B < 1 || N < 2 || pmax < 1 || pmax > N || num < 1 || rmax < 2) return 0;
  if (basis != PP_BASIS_NATURAL && basis != PP_BASIS_RAMANUJAN) return 0;
  if (kind == PP_QO_KIND_MURESAN) return (size_t)muresan_piece(B, pmax) * muresan_piece_bytes(pmax) + 256;
  if (kind != PP_QO_KIND_FIND && kind != PP_QO_KIND_SOLVE && kind != PP_QO_KIND_SOLVE_RAMANUJAN) return 0;
  if (kind == PP_QO_KIND_SOLVE_RAMANUJAN && basis != PP_BASIS_RAMANUJAN) return 0;
  DeviceFacts f;
  if (device_facts(f)) return 0;
  int rmax_eff = (rmax + kCb - 1) / kCb * kCb;
  const int cap = device_rows(f);
  if (rmax_eff > cap) rmax_eff = cap;
  const bool find = kind == PP_QO_KIND_FIND, ram = basis == PP_BASIS_RAMANUJAN;
  LongQo q;
  size_t piece = (size_t)l2_bytes() / 2 / ((size_t)long_ldr(N) * 8);
  if (piece < 1) piece = 1;
  if (piece > (size_t)B) piece = (size_t)B;
  const size_t one = long_qo_carve(find, 1, N, pmax, num, rmax_eff, ram, 0, nullptr, 0, q);
  const size_t by_budget = factor_budget / (q.l_len * 8 + 1);
  if (by_budget < piece) piece = by_budget < 1 ? 1 : by_budget;
  if (piece <= 1) return one;
  return long_qo_carve(find, (int)piece, N, pmax, num, rmax_eff, ram, 0, nullptr, 0, q);
}

int pp_long_qo_find_periods(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t num, double thresh,
                            int32_t pmin, int32_t pmax, int32_t trunc, int32_t refine, int32_t basis, const int32_t* phi,
                            int32_t table_pmax, int32_t rmax, uint32_t* periods, double* norms, int32_t* n_periods,
                            int32_t* dict_q, int32_t* dict_keep, int32_t* n_dict, int32_t* n_weights, double* weights,
                            int64_t ldw, double* res, int32_t* status, void* workspace, size_t workspace_bytes,
                            void* stream) {
  if (B == 0) return 0;
  if (int rc = check_qo_long(x, ldx, B, N, num, pmax, rmax, phi, table_pmax)) return rc;
  if (num > 64) return fail(-1, "need num <= 64%s");
  if (pmin < 1 || pmin > pmax) return fail(-1, "need 1 <= pmin <= pmax%s");
  if (refine < 0 || refine > 4) return fail(-1, "refine must be in [0, 4]%s");
  if (basis != PP_BASIS_NATURAL && basis != PP_BASIS_RAMANUJAN) return fail(-1, "unknown basis%s");
  if (!periods || !norms || !n_periods || !dict_q || !dict_keep || !n_dict || !n_weights || !weights || !status)
    return fail(-1, "output pointers are null%s");
  cudaStream_t s = (cudaStream_t)stream;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  const bool ram = basis == PP_BASIS_RAMANUJAN;
  LongQo q;
  int rmax_eff = 0;
  if (int rc = prepare(f, rmax, true, B, N, pmax, num, ram, workspace, workspace_bytes, q, rmax_eff)) return rc;
  if (ldw < q.pl.rmax) return fail(-1, "ldw must be >= rmax rounded up to a multiple of 32%s");
  const size_t smem = long_qo_smem(q.pl.wv_len());
  if (int rc = ram ? prep_kernel(long_qo_step_kernel<1>, smem, f) : prep_kernel(long_qo_step_kernel<0>, smem, f))
    return rc;
  QoOut o{periods, norms, n_periods, dict_q, dict_keep, n_dict, n_weights, weights, nullptr, ldw, res, status};
  LongQoArgs a = long_qo_args(q, x, ldx, nullptr, N, num, pmin, pmax, trunc, refine, thresh, phi);
  const LongWs& w = q.w;
  for (int b0 = 0; b0 < B; b0 += w.piece) {
    const int nw = B - b0 < w.piece ? B - b0 : w.piece;
    a.b0 = b0;
    long_load_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(x + (size_t)b0 * ldx, ldx, nw, N, w.res, w.ldr, w.sd);
    long_qo_init_kernel<<<step_grid(w, nw), kThreads, 0, s>>>(a, o, nw);
    if (int rc = check_cuda(cudaGetLastError(), "long_qo_init_kernel launch")) return rc;
    for (int round = 0; round < num; ++round) {
      int nact = 0;
      if (int rc = active_windows(w, nw, s, nact)) return rc;
      if (nact == 0) break;
      if (int rc = launch_sweep(w, N, pmin, pmax, pmax - pmin + 1, false, PP_METRIC_GAMMA, trunc, 0, nullptr, nullptr,
                                f, s))
        return rc;
      if (ram)
        long_qo_step_kernel<1><<<step_grid(w, nact), kThreads, smem, s>>>(a, o, round);
      else
        long_qo_step_kernel<0><<<step_grid(w, nact), kThreads, smem, s>>>(a, o, round);
      if (int rc = check_cuda(cudaGetLastError(), "long_qo_step_kernel launch")) return rc;
    }
  }
  return check_cuda(cudaStreamSynchronize(s), "cudaStreamSynchronize");
}

int pp_long_qo_solve(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t* periods,
                     const int32_t* nper, int32_t pmax, int32_t refine, const int32_t* phi, int32_t table_pmax,
                     int32_t rmax, const int32_t* order, int32_t n_order, int32_t* dict_q, int32_t* dict_keep,
                     int32_t* n_dict, int32_t* n_weights, double* weights, int64_t ldw, const int64_t* weights_off,
                     double* res, int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;
  if (int rc = check_qo_long(x, ldx, B, N, kmax, pmax, rmax, phi, table_pmax)) return rc;
  if (!periods || !nper || !dict_q || !dict_keep || !n_dict || !n_weights || !weights || !status)
    return fail(-1, "pointers are null%s");
  QoOut o{nullptr, nullptr, nullptr, dict_q, dict_keep, n_dict, n_weights, weights, weights_off, ldw, res, status};
  return long_qo_solve_launch(x, ldx, B, N, kmax, periods, nullptr, nper, pmax, refine, phi, rmax, order, n_order, o,
                              workspace, workspace_bytes, (cudaStream_t)stream);
}

int pp_long_qo_solve_ramanujan(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t* periods,
                               const int32_t* nper, int32_t pmax, int32_t refine, const int32_t* phi, int32_t table_pmax,
                               int32_t rmax, const int32_t* order, int32_t n_order, int32_t* dict_q, int32_t* dict_keep,
                               int32_t* n_dict, int32_t* n_weights, double* weights, int64_t ldw,
                               const int64_t* weights_off, double* res, int32_t* status, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;
  if (int rc = check_qo_long(x, ldx, B, N, kmax, pmax, rmax, phi, table_pmax)) return rc;
  if (!periods || !nper || !dict_q || !dict_keep || !n_dict || !n_weights || !weights || !status)
    return fail(-1, "pointers are null%s");
  QoOut o{nullptr, nullptr, nullptr, dict_q, dict_keep, n_dict, n_weights, weights, weights_off, ldw, res, status};
  return long_qo_solve_launch(x, ldx, B, N, kmax, periods, nullptr, nper, pmax, refine, phi, rmax, order, n_order, o,
                              workspace, workspace_bytes, (cudaStream_t)stream, true);
}

int pp_long_qo_solve_rows(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t* dict_q,
                          const int32_t* dict_rows, const int32_t* n_dict, int32_t pmax, int32_t refine, int32_t rmax,
                          int32_t* n_weights, double* weights, int64_t ldw, double* res, int32_t* status,
                          void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;
  if (int rc = check_qo_long(x, ldx, B, N, kmax, pmax, rmax, nullptr, -1)) return rc;
  if (!dict_q || !dict_rows || !n_dict || !n_weights || !weights || !status) return fail(-1, "pointers are null%s");
  QoOut o{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, n_weights, weights, nullptr, ldw, res, status};
  return long_qo_solve_launch(x, ldx, B, N, kmax, dict_q, dict_rows, n_dict, pmax, refine, nullptr, rmax, nullptr, 0, o,
                              workspace, workspace_bytes, (cudaStream_t)stream);
}

int pp_long_muresan_powers(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t max_p, int32_t normalize,
                           const int32_t* mu, int32_t table_pmax, double* raw, double* pows, int32_t* best,
                           void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;
  if (!x || !best || !mu || B < 0 || N < 2 || ldx < 1) return fail(-1, "bad arguments%s");
  if (max_p < 2 || max_p > N || table_pmax < max_p - 1) return fail(-1, "need 2 <= max_p <= N and a Moebius table covering max_p - 1%s");
  cudaStream_t s = (cudaStream_t)stream;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  const int piece = muresan_piece(B, max_p);
  if (workspace == nullptr || workspace_bytes < (size_t)piece * muresan_piece_bytes(max_p))
    return fail(-3, "workspace too small (see pp_long_qo_workspace_bytes)%s");
  double* rw = reinterpret_cast<double*>(workspace);
  const int grid = f.sm_count * kLongCtasPerSm;
  for (int b0 = 0; b0 < B; b0 += piece) {
    const int nw = B - b0 < piece ? B - b0 : piece;
    long_muresan_raw_kernel<<<grid, kThreads, 0, s>>>(x, ldx, b0, nw, N, max_p, rw, raw);
    long_muresan_final_kernel<<<nw < grid ? nw : grid, kThreads, 0, s>>>(rw, b0, nw, max_p, normalize, mu, raw, pows,
                                                                         best);
    if (int rc = check_cuda(cudaGetLastError(), "long_muresan kernels launch")) return rc;
  }
  return 0;
}

}  // extern "C"
