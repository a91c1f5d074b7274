// pyperiod_b200 -- the per-window QOPeriods solve (dictionary layout, normal equations, reconstruction) shared by
// the on-chip kernels of pp_qo.cu and the global-memory path of pp_long_qo.cu.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pyperiod_b200.h"
#include "pp_common.cuh"
#include "pp_sweep.cuh"
#include "pp_chol.cuh"
#include "pp_cg.cuh"

namespace pp {

#ifndef PP_QO_CTAS
#define PP_QO_CTAS 2
#endif
constexpr int kQoCtasPerSm = PP_QO_CTAS;  // persistent CTAs per SM of the QO kernels

struct QoPlan {
  int xs_len, n_even, rmax, num, seen_words, hier_len;
  int x0_len;   // doubles of shared memory for the original window: n_even, or 0 when it is read in place from global
  int u_len;    // Ramanujan basis: a second window-sized vector (A^T p of the conjugate gradients), else 0
  int cg_len;   // Ramanujan basis: num * pmax, the longest dictionary (rows) and the longest table set (sum of q)
  __host__ __device__ size_t off_x0() const { return (size_t)xs_len * 8; }
  __host__ __device__ size_t off_wv() const { return off_x0() + (size_t)x0_len * 8; }
  __host__ __device__ int wv_len() const { return rmax + 2 * kCb; }
  __host__ __device__ size_t off_u() const { return off_wv() + (size_t)wv_len() * 8; }
  __host__ __device__ size_t off_chol() const { return off_u() + (size_t)u_len * 8; }
  // diagonal-block scratch of the Cholesky and the hierarchical-sweep scratch are never live together
  __host__ __device__ size_t chol_bytes() const {
    const size_t a = kCholStageD;
    const size_t b = (size_t)kWarps * hier_len * 8;
    return ((a > b ? a : b) + 15) & ~(size_t)15;
  }
  __host__ __device__ size_t off_red() const { return off_chol() + chol_bytes(); }
  __host__ __device__ size_t off_bar() const { return off_red() + 2 * kWarps * 8; }
  __host__ __device__ size_t off_sweep() const { return off_bar() + 16; }
  __host__ __device__ size_t off_ints() const { return off_sweep() + ((sizeof(SweepShared) + 15) & ~15); }
  // ints: found[num] dict_q[num] dict_keep[num] dict_rows[num] dict_off[num+1] prev_rows[2 num] seen[seen_words] misc[16]
  //       tab_off[num+1]
  __host__ __device__ size_t bytes() const { return off_ints() + (size_t)(8 * num + 2 + seen_words + 16) * 4 + 16; }
  // per-CTA global workspace: packed factor (natural basis) or the conjugate-gradient vectors and Ramanujan-sum
  // tables (Ramanujan basis: c_q | fold / z | r | p | G p | w, cg_len doubles each) | saved weights | round norms
  __host__ __device__ size_t ws_L() const { return cg_len ? (size_t)6 * cg_len * 8 : chol_packed_len(rmax) * 8; }
  __host__ __device__ size_t ws_save() const { return (size_t)wv_len() * 8; }
  __host__ __device__ size_t ws_norms() const { return (((size_t)num * 8) + 255) & ~(size_t)255; }
  __host__ __device__ size_t ws_per_cta() const { return ws_L() + ws_save() + ws_norms(); }
};

__host__ __device__ inline QoPlan make_qo_plan(int N, int pmax, int num, int rmax, bool hier, bool ram_basis = false,
                                               bool x0_global = false) {
  QoPlan pl;
  pl.u_len = ram_basis ? ((N + 1) & ~1) : 0;
  pl.cg_len = ram_basis ? ((num * pmax + 31) & ~31) : 0;
  // the residual buffer doubles as the staging area of the factorisation (it is dead during a solve)
  const int stage_len = (int)(kCholStageBs / 8);
  pl.xs_len = (N + kSweepPad + 1) & ~1;
  if (pl.xs_len < stage_len) pl.xs_len = stage_len;
  pl.n_even = (N + 1) & ~1;
  pl.x0_len = x0_global ? 0 : pl.n_even;
  pl.rmax = (rmax + kCb - 1) / kCb * kCb;
  pl.num = num;
  pl.seen_words = (pmax + 32) / 32;
  pl.hier_len = hier ? hier_scratch_len(pmax) : 0;
  return pl;
}

// ------------------------------------------------------------------------------------------
// dictionary layout + normal equations + solve + reconstruction for one window
// ------------------------------------------------------------------------------------------
struct QoCtx {
  int N, num, rmax, refine;
  const int32_t* phi;   // device table, Euler phi for 0..table_pmax
  const double* x0;     // original data (shared)
  double* xs;           // residual out (shared, zero padded); staging area during the factorisation
  double* wv;           // W -> L^-1 W -> weights (shared, rmax + 64)
  double* red;
  int* found;           // periods in the order found (duplicates allowed)
  int* dict_q;          // dictionary: first-occurrence order
  int* dict_keep;       // value stored in the reference's basis_dictionary (0 for a repeated period)
  int* dict_rows;       // rows actually present in A (keep, or q when keep == 0: `if keep:` QOPeriods.py:972)
  int* dict_off;        // row offsets, [ndict+1]
  int* prev_rows;       // dict_rows of the round whose Cholesky factor is still in L (incremental factorisation)
  uint32_t* seen;       // bitmap of divisors already counted
  int seen_words;
  int* misc;            // [0]=ndict [1]=R [3]=layout scratch [8]=entries and [9]=rows of the factor held in L [10]=row_lo
  double* L;            // global, packed factor (pp_chol.cuh)
  double* wsave;        // global, rmax + 64: weights before the refinement step
  double* u;            // shared, N (Ramanujan basis only): A^T p of the conjugate gradients
  int* tab_off;         // [ndict+1] (Ramanujan basis only): first table entry of dictionary entry k (prefix sums of q)
  int cg_len;
  CholStage cs;
  long long* t;         // per-thread phase timers (development aid): [0] layout [1] W + tables [2] factor [3] solves
};

// QOPeriods.get_subspaces (QOPeriods.py:830-840) for `found[0..nfound)`.  All threads call (contains
// barriers): the divisor scan of each period is spread over the CTA, the bookkeeping is thread 0's.
__device__ inline void qo_layout(const QoCtx& c, int nfound) {
  const int tid = threadIdx.x;
  for (int i = tid; i < c.seen_words; i += kThreads) c.seen[i] = 0u;
  if (tid == 0) c.misc[0] = 0;
  __syncthreads();
  for (int f = 0; f < nfound; ++f) {
    const int q = c.found[f];
    if (tid == 0) c.misc[3] = 0;
    __syncthreads();
    int fresh = 0;
    for (int d = 1 + tid; d <= q; d += kThreads) {
      if (q % d == 0 && !((c.seen[d >> 5] >> (d & 31)) & 1u)) {
        fresh += c.phi[d];
        atomicOr(&c.seen[d >> 5], 1u << (d & 31));
      }
    }
    if (fresh) atomicAdd(&c.misc[3], fresh);
    __syncthreads();
    if (tid == 0) {
      int ndict = c.misc[0], slot = -1;
      for (int k = 0; k < ndict; ++k)
        if (c.dict_q[k] == q) slot = k;
      if (slot < 0) slot = ndict++;
      c.dict_q[slot] = q;
      c.dict_keep[slot] = c.misc[3];   // a repeated period overwrites its entry with 0 new dimensions
      c.misc[0] = ndict;
    }
    __syncthreads();
  }
  if (tid == 0) {
    const int ndict = c.misc[0];
    int off = 0;
    for (int k = 0; k < ndict; ++k) {
      c.dict_rows[k] = c.dict_keep[k] ? c.dict_keep[k] : c.dict_q[k];
      c.dict_off[k] = off;
      off += c.dict_rows[k];
    }
    c.dict_off[ndict] = off;
    c.misc[1] = off;
  }
}

// fold sums of src over the kept rows of the dictionary: out[row] = sum_{n = i (mod q)} src[n], terms in increasing n
// (W = A x, QOPeriods.py:782).  No barrier inside.
__device__ __forceinline__ void qo_fold_rows(const QoCtx& c, int ndict, const double* src, double* out) {
  for (int k = 0; k < ndict; ++k) {
    const int q = c.dict_q[k], rows = c.dict_rows[k], off = c.dict_off[k];
    for (int i = threadIdx.x; i < rows; i += kThreads) {
      double s = 0.0;
      for (int n = i; n < c.N; n += q) s += src[n];
      out[off + i] = s;
    }
  }
}

// xs = x0 - A^T w, returns sum of squares of the reconstruction A^T w (to every thread).  Contains barriers.
__device__ __forceinline__ double qo_reconstruct(const QoCtx& c, int ndict) {
  double e = 0.0;
  for (int n = threadIdx.x; n < c.N; n += kThreads) {
    double r = 0.0;
    for (int k = 0; k < ndict; ++k) {
      const int i = n % c.dict_q[k];
      if (i < c.dict_rows[k]) r += c.wv[c.dict_off[k] + i];
    }
    c.xs[n] = c.x0[n] - r;
    e = fma(r, r, e);
  }
  e = warp_sum(e);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) c.red[threadIdx.x >> 5] = e;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < kWarps; ++w) t += c.red[w];
  __syncthreads();
  return t;
}

// Returns 0 ok, PP_STATUS_SINGULAR, PP_STATUS_TOO_LARGE.  On success wv holds the weights, xs the residual,
// and *e_recon the sum of squares of the reconstruction.  All threads call; contains barriers.
__device__ inline int cta_qo_solve(const QoCtx& c, int nfound, double* e_recon, bool explicit_layout = false) {
  const int tid = threadIdx.x;
  const int N = c.N;
  long long tm = clock64();
  // explicit_layout: the caller has filled dict_q / dict_rows / dict_off and misc[0] (entries), misc[1] (rows)
  if (!explicit_layout) qo_layout(c, nfound);
  __syncthreads();
  { const long long now = clock64(); c.t[0] += now - tm; tm = now; }
  const int ndict = c.misc[0], R = c.misc[1];
  // more rows than samples: A A^T has rank <= N < R, the normal equations are singular
  if (R > N) return PP_STATUS_SINGULAR;
  if (R > c.rmax) return PP_STATUS_TOO_LARGE;
  if (R == 0) {
    for (int n = tid; n < N; n += kThreads) c.xs[n] = c.x0[n];
    __syncthreads();
    *e_recon = 0.0;
    return PP_STATUS_OK;
  }
  // The dictionary only grows from round to round (unless a repeated period rewrites an entry), so the factor of
  // the previous round is the leading block of this round's: only the rows from the last 32-aligned boundary on
  // are computed (the partial block below it is redone from its integer counts).
  if (tid == 0) {
    const int nd_prev = c.misc[8], r_prev = c.misc[9];
    bool grow = r_prev > 0 && ndict >= nd_prev;
    for (int k = 0; grow && k < nd_prev; ++k) grow = c.dict_rows[k] == c.prev_rows[k] && c.dict_q[k] == c.prev_rows[c.num + k];
    c.misc[10] = grow ? (r_prev / kCb) * kCb : 0;
    c.misc[9] = 0;  // no valid factor until this round's succeeds
  }
  const DictView dv{c.dict_q, c.dict_rows, c.dict_off, ndict, N};
  qo_fold_rows(c, ndict, c.x0, c.wv);   // W = A x, of the ORIGINAL data
  const int Rpad = (R + kCb - 1) / kCb * kCb + kCb;
  for (int i = R + tid; i < Rpad; i += kThreads) c.wv[i] = 0.0;
  __syncthreads();
  const int row_lo = c.misc[10];
  { const long long now = clock64(); c.t[1] += now - tm; tm = now; }
  if (!cta_chol_factor(c.L, R, row_lo, dv, c.wv, c.cs, c.t + 4)) return PP_STATUS_SINGULAR;
  if (tid == 0) {  // L now holds the factor of this dictionary
    c.misc[8] = ndict;
    c.misc[9] = R;
    for (int k = 0; k < ndict; ++k) {
      c.prev_rows[k] = c.dict_rows[k];
      c.prev_rows[c.num + k] = c.dict_q[k];
    }
  }
  { const long long now = clock64(); c.t[2] += now - tm; tm = now; }
  cta_chol_backward(c.L, R, c.wv, c.cs);
  double e = qo_reconstruct(c, ndict);
  // Iterative refinement with the implicit Gram product: G w = A (A^T w), so the residual of the normal equations is
  // the fold of the signal residual, W - G w = A (x - A^T w).  `refine` steps are always taken; while a step still
  // moves the weights by more than 1e-11 of their size (an ill-conditioned dictionary) and the corrections keep
  // shrinking, up to four more follow.
  double prev_step = 0.0;
  const int max_steps = c.refine > 0 ? c.refine + 4 : 0;
  for (int it = 0; it < max_steps; ++it) {
    for (int i = tid; i < Rpad; i += kThreads) c.wsave[i] = c.wv[i];
    __syncthreads();
    qo_fold_rows(c, ndict, c.xs, c.wv);
    __syncthreads();
    cta_chol_forward(c.L, R, c.wv, c.cs);
    cta_chol_backward(c.L, R, c.wv, c.cs);
    double dmax = 0.0, wmax = 0.0;
    for (int i = tid; i < R; i += kThreads) {
      dmax = fmax(dmax, fabs(c.wv[i]));
      wmax = fmax(wmax, fabs(c.wsave[i]));
    }
    dmax = warp_max(dmax);
    wmax = warp_max(wmax);
    __syncthreads();
    if ((tid & 31) == 0) {
      c.red[tid >> 5] = dmax;
      c.red[kWarps + (tid >> 5)] = wmax;
    }
    __syncthreads();
    dmax = wmax = 0.0;
    for (int w = 0; w < kWarps; ++w) {
      dmax = fmax(dmax, c.red[w]);
      wmax = fmax(wmax, c.red[kWarps + w]);
    }
    __syncthreads();
    const bool diverging = it > 0 && !(dmax < 0.5 * prev_step);   // uniform
    if (diverging && it >= c.refine) {
      // the correction stopped shrinking: keep the weights of the previous step
      for (int i = tid; i < R; i += kThreads) c.wv[i] = c.wsave[i];
      __syncthreads();
      e = qo_reconstruct(c, ndict);
      break;
    }
    for (int i = tid; i < R; i += kThreads) c.wv[i] += c.wsave[i];
    __syncthreads();
    e = qo_reconstruct(c, ndict);
    prev_step = dmax;
    if (it + 1 >= c.refine && !(dmax > 1e-11 * wmax)) break;
  }
  c.t[3] += clock64() - tm;
  *e_recon = e;
  return PP_STATUS_OK;
}

// ------------------------------------------------------------------------------------------
// basis_type = "ramanujan" (QOPeriods.py:970-971, 1005-1052): row i of period q is c_q((n - i) mod q), n < N
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int mobius_int(int m) {
  int res = 1;
  for (int d = 2; d * d <= m; ++d) {
    if (m % d == 0) {
      m /= d;
      if (m % d == 0) return 0;
      res = -res;
    }
  }
  return m > 1 ? -res : res;
}

// The Ramanujan-sum dictionary applied implicitly: A u is a fold of u per period followed by a circular
// correlation with c_q, A^T v a circular convolution per period followed by a tiling.
struct RamBasisOp {
  int nd, N;
  const int* dq;
  const int* drows;
  const int* doff;    // first row of entry k
  const int* toff;    // first table element of entry k
  const double* cq;   // global: c_q tables (exact integers)
  double* fold;       // global scratch, sum of q
  __device__ void apply(const double* u, double* out) const {
    for (int k = 0; k < nd; ++k) {
      const int q = dq[k];
      double* f = fold + toff[k];
      for (int m = threadIdx.x; m < q; m += kThreads) {
        double s = 0.0;
        for (int n = m; n < N; n += q) s += u[n];
        f[m] = s;
      }
    }
    __syncthreads();
    for (int k = 0; k < nd; ++k) {
      const int q = dq[k], rows = drows[k];
      const double* f = fold + toff[k];
      const double* c = cq + toff[k];
      for (int i = threadIdx.x; i < rows; i += kThreads) {
        int idx = i == 0 ? 0 : q - i;   // (0 - i) mod q
        double s0 = 0.0, s1 = 0.0;
        int m = 0;
        for (; m + 1 < q; m += 2) {
          s0 = fma(c[idx], f[m], s0);
          if (++idx == q) idx = 0;
          s1 = fma(c[idx], f[m + 1], s1);
          if (++idx == q) idx = 0;
        }
        if (m < q) s0 = fma(c[idx], f[m], s0);
        out[doff[k] + i] = s0 + s1;
      }
    }
  }
  __device__ void apply_t(const double* v, double* out) const {
    for (int k = 0; k < nd; ++k) {
      const int q = dq[k], rows = drows[k];
      double* z = fold + toff[k];
      const double* c = cq + toff[k];
      const double* vk = v + doff[k];
      for (int m = threadIdx.x; m < q; m += kThreads) {
        int idx = m;   // (m - i) mod q
        double s0 = 0.0, s1 = 0.0;
        int i = 0;
        for (; i + 1 < rows; i += 2) {
          s0 = fma(vk[i], c[idx], s0);
          idx = idx == 0 ? q - 1 : idx - 1;
          s1 = fma(vk[i + 1], c[idx], s1);
          idx = idx == 0 ? q - 1 : idx - 1;
        }
        if (i < rows) s0 = fma(vk[i], c[idx], s0);
        z[m] = s0 + s1;
      }
    }
    __syncthreads();
    for (int n = threadIdx.x; n < N; n += kThreads) {
      double s = 0.0;
      for (int k = 0; k < nd; ++k) s += fold[toff[k] + n % dq[k]];
      out[n] = s;
    }
  }
};

// Same contract as cta_qo_solve for the Ramanujan-sum dictionary.  Its Gram matrix is singular by construction (q
// shifted rows span phi(q) dimensions); the reference's np.linalg.solve runs on the rounding-perturbed matrix and
// its reconstruction is the orthogonal projection onto the row space to 1e-14, which is what conjugate gradients
// deliver here (pp_cg.cuh).  The weights returned are the minimum-norm solution (the reference's are whatever its LU
// produced; only A^T w is determined).
__device__ inline int cta_qo_solve_ram(const QoCtx& c, int nfound, double* e_recon) {
  const int tid = threadIdx.x;
  const int N = c.N;
  long long tm = clock64();
  qo_layout(c, nfound);
  __syncthreads();
  { const long long now = clock64(); c.t[0] += now - tm; tm = now; }
  const int ndict = c.misc[0], R = c.misc[1];
  // The one EXACT singularity of this dictionary: both rows of period 2 (+1 -1 +1 ... and its negative; cos(pi) is
  // exactly -1 in the reference's sum of exponentials, QOPeriods.py:1037-1045).  Two exactly opposite rows make the
  // reference's LU hit a zero pivot: np.linalg.solve raises LinAlgError and the loop keeps the previous round
  // (:552-559).  Every other dependency of the Ramanujan rows is perturbed by ~1e-13 of rounding and goes through.
  for (int k = 0; k < ndict; ++k)
    if (c.dict_q[k] == 2 && c.dict_rows[k] == 2) return PP_STATUS_SINGULAR;
  if (R > c.rmax) return PP_STATUS_TOO_LARGE;
  for (int n = tid; n < N; n += kThreads) c.xs[n] = c.x0[n];
  if (tid == 0) {
    int off = 0;
    for (int k = 0; k < ndict; ++k) {
      c.tab_off[k] = off;
      off += c.dict_q[k];
    }
    c.tab_off[ndict] = off;
  }
  __syncthreads();
  if (R == 0) {
    *e_recon = 0.0;
    return PP_STATUS_OK;
  }
  double* cq = c.L;
  double* fold = c.L + c.cg_len;
  double* r = c.L + 2 * (size_t)c.cg_len;
  double* p = c.L + 3 * (size_t)c.cg_len;
  double* ap = c.L + 4 * (size_t)c.cg_len;
  double* w = c.L + 5 * (size_t)c.cg_len;
  for (int k = 0; k < ndict; ++k) {
    const int q = c.dict_q[k], phq = c.phi[q];
    for (int m = tid; m < q; m += kThreads) {
      int a = q, bb = m;   // gcd(m, q), gcd(0, q) = q
      while (bb) {
        const int t = a % bb;
        a = bb;
        bb = t;
      }
      const int qg = q / a;
      cq[c.tab_off[k] + m] = (double)(mobius_int(qg) * (phq / c.phi[qg]));   // c_q(m) = mu(q/g) phi(q) / phi(q/g)
    }
  }
  for (int i = tid; i < R; i += kThreads) w[i] = 0.0;
  __syncthreads();
  { const long long now = clock64(); c.t[1] += now - tm; tm = now; }
  RamBasisOp op{ndict, N, c.dict_q, c.dict_rows, c.dict_off, c.tab_off, cq, fold};
  // Budget per pass: R + 16 steps, as gp_kernel.  In exact arithmetic CG ends within rank(G) <= R steps; a fixed
  // budget below that restarts the pass and discards the Krylov space (1365, 1364, 1024 at N = 4096: about 1040
  // steps in one pass, no convergence in four passes of 500).
  const int steps = cta_cg_project(op, R, N, c.xs, c.u, r, p, ap, w, c.red, R + 16);
  __syncthreads();
  if (steps < 0) return PP_STATUS_GUARD;
  for (int i = tid; i < R; i += kThreads) c.wv[i] = w[i];
  double e = 0.0;
  for (int n = tid; n < N; n += kThreads) {
    const double rr = c.x0[n] - c.xs[n];
    e = fma(rr, rr, e);
  }
  e = warp_sum(e);
  __syncthreads();
  if ((tid & 31) == 0) c.red[tid >> 5] = e;
  __syncthreads();
  double t = 0.0;
  for (int wv = 0; wv < kWarps; ++wv) t += c.red[wv];
  __syncthreads();
  c.t[3] += clock64() - tm;
  *e_recon = t;
  return PP_STATUS_OK;
}

struct QoOut {
  uint32_t* periods;   // [B, num]  periods reported (found order)
  double* norms;       // [B, num]
  int32_t* n_periods;  // [B] number reported (may be one less than the dictionary holds, QOPeriods.py:585-588)
  int32_t* dict_q;     // [B, num]
  int32_t* dict_keep;  // [B, num]
  int32_t* n_dict;     // [B]
  int32_t* n_weights;  // [B]
  double* weights;     // window b: weights + (weights_off ? weights_off[b] : b * ldw)
  const int64_t* weights_off;
  int64_t ldw;
  double* res;         // [B, N] (nullable)
  int32_t* status;     // [B]
  // overflow pool of the find kernel (nullable): a window whose dictionary outgrows the ldw doubles of its inline
  // row takes one slot of pool_stride doubles; pool_slot[b] = its index, or -1
  double* pool = nullptr;
  int pool_slots = 0;
  int64_t pool_stride = 0;
  int* pool_counter = nullptr;
  int32_t* pool_slot = nullptr;
  __device__ double* weights_of(int b) const { return weights + (weights_off ? weights_off[b] : (int64_t)b * ldw); }
};

// Writes the outputs of a solved round.  Returns false (uniformly, nothing written) when the weights need a pool slot
// and the pool is exhausted.  misc[11]: pool slot of this window (-1: none yet).  Contains a barrier when a pool is
// in use.
__device__ inline bool qo_commit(const QoCtx& c, const QoOut& o, int b, int nfound, const double* round_norms) {
  const int tid = threadIdx.x;
  const int ndict = c.misc[0], R = c.misc[1];
  double* w = o.weights_of(b);
  if (o.pool != nullptr) {
    if (R > o.ldw) {
      if (tid == 0 && c.misc[11] < 0) c.misc[11] = atomicAdd(o.pool_counter, 1);
      __syncthreads();
      const int slot = c.misc[11];
      if (slot >= o.pool_slots) return false;
      w = o.pool + (size_t)slot * o.pool_stride;
    }
    if (tid == 0) o.pool_slot[b] = (R > o.ldw) ? c.misc[11] : -1;
  }
  for (int i = tid; i < c.num; i += kThreads) {
    o.periods[(size_t)b * c.num + i] = i < nfound ? (uint32_t)c.found[i] : 0u;
    o.norms[(size_t)b * c.num + i] = i < nfound ? round_norms[i] : 0.0;
    o.dict_q[(size_t)b * c.num + i] = i < ndict ? c.dict_q[i] : 0;
    o.dict_keep[(size_t)b * c.num + i] = i < ndict ? c.dict_keep[i] : 0;
  }
  for (int i = tid; i < R; i += kThreads) w[i] = c.wv[i];
  if (o.res)
    for (int n = tid; n < c.N; n += kThreads) o.res[(size_t)b * c.N + n] = c.xs[n];
  if (tid == 0) {
    o.n_periods[b] = nfound;
    o.n_dict[b] = ndict;
    o.n_weights[b] = R;
  }
  return true;
}

__device__ __forceinline__ QoCtx make_ctx(unsigned char* smem, const QoPlan& pl, int N, int num, int refine,
                                          const int32_t* phi, unsigned char* ws_cta) {
  QoCtx c;
  c.N = N;
  c.num = num;
  c.rmax = pl.rmax;
  c.refine = refine;
  c.phi = phi;
  c.xs = reinterpret_cast<double*>(smem);
  c.x0 = reinterpret_cast<double*>(smem + pl.off_x0());
  c.wv = reinterpret_cast<double*>(smem + pl.off_wv());
  c.u = reinterpret_cast<double*>(smem + pl.off_u());
  c.cg_len = pl.cg_len;
  double* chol = reinterpret_cast<double*>(smem + pl.off_chol());
  c.cs.Bs = c.xs;  // the residual buffer is dead while a factorisation runs
  c.cs.D = chol;
  c.cs.Li = chol + kCb * kLdD;
  c.cs.rD = c.cs.Li + kCb * kLdD;
  c.cs.flag = reinterpret_cast<int*>(c.cs.rD + kCb);
  c.red = reinterpret_cast<double*>(smem + pl.off_red());
  int* ints = reinterpret_cast<int*>(smem + pl.off_ints());
  c.found = ints;
  c.dict_q = ints + num;
  c.dict_keep = ints + 2 * num;
  c.dict_rows = ints + 3 * num;
  c.dict_off = ints + 4 * num;
  c.prev_rows = ints + 5 * num + 1;   // [2 * num]: rows, then periods
  c.seen = reinterpret_cast<uint32_t*>(ints + 7 * num + 1);
  c.seen_words = pl.seen_words;
  c.misc = ints + 7 * num + 1 + pl.seen_words;
  c.tab_off = c.misc + 16;
  c.L = reinterpret_cast<double*>(ws_cta);
  c.wsave = reinterpret_cast<double*>(ws_cta + pl.ws_L());
  c.t = nullptr;
  return c;
}

// windows of a launch: `order` (nullable) lists the window indices to process, in hand-out order
struct QoBatch {
  const double* x;
  int64_t ldx;
  int count;             // windows to process
  const int32_t* order;  // [count] or null (identity)
  __device__ int window(int i) const { return order ? order[i] : i; }
};

}  // namespace pp
