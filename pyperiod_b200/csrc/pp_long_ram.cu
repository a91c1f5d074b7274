// pyperiod_b200 -- the fp64 Ramanujan periodogram of windows whose on-chip plan does not fit in shared memory
// (the "long" path of pp_ramanujan.cu).  Same quantity, same fold order, same tensor cores; see DESIGN.md 5.9.
//
//   norms[b, q] = (q / phi(q)^2)^2 * sum_m cnt_q[m] * (H S_q)_m^2,   H[m][l] = c_q((l - m) mod q)
//
// The folds S_q and the dictionary c_q live in the workspace (L2-resident by construction) instead of shared memory.
// A batch runs as pieces of at most kLrPieceWin windows; the periods of a piece run in chunks, largest first, whose
// folds fit the fold buffer.  Per (piece, chunk), four launches on the caller's stream:
//   long_ram_cq_kernel    c_q of the chunk's periods (chunk-relative triangular offsets; nothing grows with qmax^2)
//   long_ram_fold_kernel  S_q of every window and period of the chunk, summed in increasing n as fold_all_kernel
//   long_ram_dmma_kernel  the contraction on the FP64 tensor cores (mma.sync m8n8k4 f64), one partial norm per unit
//   long_ram_reduce_kernel  the partial norms of a (window, period) added in a fixed order: runs are bit-identical
//
// Work unit of the contraction = (period, column group, block of 512 A rows).
//  * Group form (8 live windows): the A rows are the rows of H, the 8 B columns the 8 windows' folds.
//  * Shift form (a window of a group with fewer than 8 live windows, e.g. the 1-D call): residue m = 8 i + j gives
//    z[8 i + j] = sum_l c_q(l - 8 i) S_q[(l + j) mod q], so the A rows are every 8th row of H and the 8 B columns are
//    8 cyclic shifts of one window's folds.  The tensor work is q^2 per window in both forms.
// The k dimension runs in chunks of kLrK folds; each chunk's B tile and the slice of c_q its A fragments read
// (kLrK + s (rows - 1) consecutive entries mod q, s = 1 or 8) are brought in by cp.async, double-buffered.  The
// units of one period are handed out together, so its folds are read from L2.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pyperiod_b200.h"
#include "pp_common.cuh"
#include "pp_host.cuh"
#include "pp_ram.cuh"

namespace pp {
namespace {

constexpr int kLrRows = 512;                          // A rows per unit: 64 fragments, 8 per warp
constexpr int kLrFrags = kLrRows / 8 / kWarps;        // fragments per warp
constexpr int kLrK = 64;                              // folds per k-chunk
constexpr int kLrSpan = kLrK + 8 * (kLrRows - 1);     // c_q entries of a chunk's A fragments (shift form)
constexpr int kLrStage = kLrK * 8 + kLrSpan;          // doubles per stage: B tile [kLrK][8], then the c_q slice
constexpr size_t kLrSmem = (size_t)(2 * kLrStage + kWarps * 8) * 8 + 16;
constexpr int kLrPieceWin = 64;                       // windows per piece
constexpr size_t kLrFoldBudget = (size_t)64 << 20;    // bytes of folds and c_q pp_long_ramanujan_workspace_bytes
                                                      // provides for

static_assert(kLrFrags == 8, "one warp pass covers 8 fragments");
static_assert((kLrStage * 8) % 16 == 0, "stages stay 16-byte aligned");

// row blocks of period q in a form with A-row stride s (1: group form, q rows; 8: shift form, ceil(q / 8) rows)
__host__ __device__ inline int lr_blocks(int q, int s) {
  const int rows = s == 1 ? q : (q + 7) / 8;
  return (rows + kLrRows - 1) / kLrRows;
}
__host__ __device__ inline long long lr_units(int q, int gfull, int nlone) {
  return (long long)gfull * lr_blocks(q, 1) + (long long)nlone * lr_blocks(q, 8);
}
// rows of the chunk's periods below q (folds and c_q share this chunk-relative layout)
__host__ __device__ inline size_t lr_roff(int q, int qa) { return cq_offset(q) - cq_offset(qa); }

__device__ __forceinline__ void cp_async_8(void* dst_smem, const void* src, int src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(smem_u32(dst_smem)), "l"(src), "r"(src_bytes)
               : "memory");
}

// ------------------------------------------------------------------------------------------
// c_q and folds of a chunk
// ------------------------------------------------------------------------------------------
// grid: one CTA per period, q = qb - blockIdx.x
__global__ void long_ram_cq_kernel(int qa, int qb, const int32_t* __restrict__ mu, const int32_t* __restrict__ phi,
                                   double* __restrict__ cq) {
  const int q = qb - blockIdx.x;
  double* out = cq + lr_roff(q, qa);
  for (int n = threadIdx.x; n < q; n += blockDim.x) out[n] = ramanujan_sum(n, q, mu, phi);
}

// grid: (any, periods), q = qb - blockIdx.y.  Window w of the piece: group form (w < 8 gfull) rows of 8 windows,
// S[((w / 8) rc + roff + m) 8 + w % 8]; shift form one vector per window, S[8 gfull rc + (w - 8 gfull) rc + roff + m].
__global__ void __launch_bounds__(kThreads) long_ram_fold_kernel(const double* __restrict__ x, int64_t ldx, int nw,
                                                                  int gfull, int N, int qa, int qb,
                                                                  double* __restrict__ S, size_t rc) {
  const int q = qb - blockIdx.y;
  const size_t ro = lr_roff(q, qa);
  const int items = q * nw;
  for (int idx = blockIdx.x * kThreads + threadIdx.x; idx < items; idx += gridDim.x * kThreads) {
    const int w = idx / q, m = idx - w * q;   // residues fastest: the reads of a warp are contiguous
    const double* src = x + (size_t)w * ldx;
    double a = 0.0;
    for (int n = m; n < N; n += q) a += __ldg(src + n);   // increasing n, one chain, as fold_all_kernel
    if (w < 8 * gfull)
      S[((size_t)(w >> 3) * rc + ro + m) * 8 + (w & 7)] = a;
    else
      S[(size_t)gfull * 8 * rc + (size_t)(w - 8 * gfull) * rc + ro + m] = a;
  }
}

// ------------------------------------------------------------------------------------------
// contraction on the FP64 tensor cores
// ------------------------------------------------------------------------------------------
struct LongRamArgs {
  const double* S;       // folds of the piece (layout of long_ram_fold_kernel)
  const double* cq;      // c_q of the chunk
  double* part;          // [nw][nq][nrbs] partial norms
  int* counter;
  size_t rc;             // fold rows per window the buffer holds
  int qa, qb, nq, nrbs, gfull, nlone, N;
  long long units;
};

// one k-chunk of a warp: NFR fragments (A rows 8 (wid + 8 i) .. + 7 of the block) against the staged B tile.  A
// lane's A element at k-step k4 is sl[tb[i] + 4 k4]: the slice is staged per chunk, so tb is fixed over the unit.
template <int NFR>
__device__ __forceinline__ void lr_chunk(double (&acc)[kLrFrags][2], const double* __restrict__ Bs,
                                         const double* __restrict__ sl, const int (&tb)[kLrFrags]) {
  const int lane = threadIdx.x & 31, lr = lane >> 2, lc = lane & 3;
  const double* bp = Bs + lc * 8 + lr;
#pragma unroll
  for (int k4 = 0; k4 < kLrK / 4; ++k4) {
    const double b = bp[k4 * 32];
#pragma unroll
    for (int i = 0; i < NFR; ++i) dmma_m8n8k4(acc[i], sl[tb[i] + 4 * k4], b);
  }
}

// persistent grid; units handed out by a global counter: periods descending (the units of one period together),
// then the group-form column groups, then the shift-form windows, row blocks innermost.
__global__ void __launch_bounds__(kThreads, 2) long_ram_dmma_kernel(LongRamArgs a) {
  double* st0 = reinterpret_cast<double*>(pp_smem);
  double* red = st0 + 2 * kLrStage;                  // [kWarps][8]
  int* unit_slot = reinterpret_cast<int*>(red + kWarps * 8);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, lr = lane >> 2, lc = lane & 3;
  // period of the units this CTA draws: they increase, so the cursor only moves down the periods
  int cur_q = a.qb;
  long long cur_base = 0, cur_n = lr_units(cur_q, a.gfull, a.nlone);
  for (;;) {
    if (tid == 0) *unit_slot = atomicAdd(a.counter, 1);
    __syncthreads();   // also: every warp is done with the stages and red of the previous unit
    const long long u = *unit_slot;
    if (u >= a.units) break;
    while (u >= cur_base + cur_n) {
      cur_base += cur_n;
      --cur_q;
      cur_n = lr_units(cur_q, a.gfull, a.nlone);
    }
    const int q = cur_q;
    int idx = (int)(u - cur_base);
    const int nrb1 = lr_blocks(q, 1), nrb8 = lr_blocks(q, 8);
    bool shift;
    int col, rb;   // col: first window of the group (group form) or the window (shift form), piece-relative
    if (idx < a.gfull * nrb1) {
      shift = false;
      col = 8 * (idx / nrb1);
      rb = idx % nrb1;
    } else {
      idx -= a.gfull * nrb1;
      shift = true;
      col = 8 * a.gfull + idx / nrb8;
      rb = idx % nrb8;
    }
    const int s = shift ? 8 : 1;
    const int arows = shift ? (q + 7) / 8 : q;
    const int r0 = rb * kLrRows;
    const int nfb = min(kLrRows / 8, (arows - r0 + 7) / 8);   // fragments of this block
    const int ra = 8 * nfb;
    const int span = kLrK + s * (ra - 1);
    const int nfr = max(0, (nfb - wid + 7) / 8);               // fragments of this warp: wid, wid + 8, ...
    const size_t ro = lr_roff(q, a.qa);
    const double* cqq = a.cq + ro;
    const double* Sq = shift ? a.S + (size_t)a.gfull * 8 * a.rc + (size_t)(col - 8 * a.gfull) * a.rc + ro
                             : a.S + ((size_t)(col >> 3) * a.rc + ro) * 8;
    // slice of chunk l0: sl[t] = c_q((l0 - s (r0 + ra - 1) + t) mod q); A row r at column l reads t = l - l0 + s (r0 +
    // ra - 1 - r)
    const int e_first = (int)((q - (long long)s * (r0 + ra - 1) % q) % q);
    int tb[kLrFrags];
#pragma unroll
    for (int i = 0; i < kLrFrags; ++i) tb[i] = i < nfr ? lc + s * (ra - 1 - 8 * (wid + 8 * i) - lr) : 0;
    double acc[kLrFrags][2];
#pragma unroll
    for (int i = 0; i < kLrFrags; ++i) acc[i][0] = acc[i][1] = 0.0;

    auto stage = [&](double* dst, int l0) {
      if (!shift) {   // B[k][w] = S_q[l0 + k] of window w: rows of 64 bytes, zero past q
        for (int i = tid; i < kLrK * 4; i += kThreads) {
          const int k = i >> 2, c = i & 3;
          const int bytes = l0 + k < q ? 16 : 0;
          cp_async_16(dst + k * 8 + 2 * c, bytes ? Sq + (size_t)(l0 + k) * 8 + 2 * c : Sq, bytes);
        }
      } else {        // B[k][j] = S_q[(l0 + k + j) mod q], zero for l0 + k past q
        for (int i = tid; i < kLrK * 8; i += kThreads) {
          const int k = i >> 3, j = i & 7;
          int e = l0 + k + j;
          if (e >= q) e = e - q < q ? e - q : e % q;
          cp_async_8(dst + i, l0 + k < q ? Sq + e : Sq, l0 + k < q ? 8 : 0);
        }
      }
      double* sl = dst + kLrK * 8;
      int e0 = e_first + l0;   // l0 < q
      if (e0 >= q) e0 -= q;
      for (int t = tid; t < span; t += kThreads) {
        int e = e0 + t;
        if (e >= q) e = e - q < q ? e - q : e % q;
        cp_async_8(sl + t, cqq + e, 8);
      }
      cp_async_commit();
    };

    const int nk = (q + kLrK - 1) / kLrK;
    stage(st0, 0);
    for (int kc = 0; kc < nk; ++kc) {
      const double* cur = st0 + (kc & 1) * kLrStage;
      if (kc + 1 < nk) {
        stage(st0 + ((kc + 1) & 1) * kLrStage, (kc + 1) * kLrK);
        cp_async_wait<1>();
      } else {
        cp_async_wait<0>();
      }
      __syncthreads();
      const double* sl = cur + kLrK * 8;
      switch (nfr) {
        case 8: lr_chunk<8>(acc, cur, sl, tb); break;
        case 7: lr_chunk<7>(acc, cur, sl, tb); break;
        case 6: lr_chunk<6>(acc, cur, sl, tb); break;
        case 5: lr_chunk<5>(acc, cur, sl, tb); break;
        case 4: lr_chunk<4>(acc, cur, sl, tb); break;
        case 3: lr_chunk<3>(acc, cur, sl, tb); break;
        case 2: lr_chunk<2>(acc, cur, sl, tb); break;
        case 1: lr_chunk<1>(acc, cur, sl, tb); break;
        default: break;
      }
      __syncthreads();   // everyone is done with this stage before it is refilled
    }
    // cnt-weighted squares of this lane's outputs: D[r][2 lc + e] is residue r (group form, window 2 lc + e) or
    // 8 r + 2 lc + e (shift form); fragments past nfr hold zeros
    const int Mrows = a.N / q, rq = a.N - Mrows * q;
    double c[2] = {0.0, 0.0};
#pragma unroll
    for (int i = 0; i < kLrFrags; ++i) {
      const int r = r0 + 8 * (wid + 8 * i) + lr;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int m = shift ? 8 * r + 2 * lc + e : r;
        const double cnt = m < q ? (double)(Mrows + (m < rq ? 1 : 0)) : 0.0;
        c[e] = fma(cnt * acc[i][e], acc[i][e], c[e]);
      }
    }
    // over the 8 row-lanes, then over the warps in a fixed order
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      double v = c[e];
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      c[e] = v;
    }
    if (lane < 4) {
      red[wid * 8 + 2 * lane] = c[0];
      red[wid * 8 + 2 * lane + 1] = c[1];
    }
    __syncthreads();
    const size_t qi = (size_t)(q - a.qa);
    if (!shift) {
      if (tid < 8) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) t += red[w * 8 + tid];
        a.part[((size_t)(col + tid) * a.nq + qi) * a.nrbs + rb] = t;
      }
    } else if (tid == 0) {
      double t = 0.0;
      for (int w = 0; w < kWarps; ++w)
#pragma unroll
        for (int j = 0; j < 8; ++j) t += red[w * 8 + j];
      a.part[((size_t)col * a.nq + qi) * a.nrbs + rb] = t;
    }
  }
}

// norms[w, q] = (q / phi^2)^2 * sum of the partial norms of (w, q) in ascending row-block order
__global__ void long_ram_reduce_kernel(const double* __restrict__ part, int nw, int gfull, int qa, int nq, int nrbs,
                                       const int32_t* __restrict__ phi, double* __restrict__ norms, int ld_norms) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= nw * nq) return;
  const int w = idx / nq, qi = idx - w * nq, q = qa + qi;
  const int nrb = lr_blocks(q, w < 8 * gfull ? 1 : 8);
  const double* p = part + ((size_t)w * nq + qi) * nrbs;
  double t = 0.0;
  for (int rb = 0; rb < nrb; ++rb) t += p[rb];
  const double ph = (double)phi[q];
  const double scale = (double)q / (ph * ph);   // C^T C = (q / phi^2) circ(c_q)
  norms[(size_t)w * ld_norms + q] = scale * scale * t;
}

// ------------------------------------------------------------------------------------------
// workspace
// ------------------------------------------------------------------------------------------
struct LongRamWs {
  int* counter = nullptr;
  double* cq = nullptr;     // [rc]       c_q of a chunk
  double* S = nullptr;      // [wp * rc]  folds of a piece and chunk
  double* part = nullptr;   // [wp * pc]  partial norms
};

static int piece_windows(int B) { return B < 1 ? 1 : (B < kLrPieceWin ? B : kLrPieceWin); }
static size_t partial_cap(size_t rc) { return rc / 128 + 64; }   // (periods x row blocks) of a chunk

// bytes of the layout for wp windows and rc fold rows; carves the pieces when ws holds them
static size_t long_ram_layout(void* ws, size_t ws_bytes, int wp, size_t rc, LongRamWs* out) {
  const size_t sizes[4] = {256, rc * 8, (size_t)wp * rc * 8, (size_t)wp * partial_cap(rc) * 8};
  size_t off = 0, at[4];
  for (int i = 0; i < 4; ++i) {
    off = (off + 255) & ~(size_t)255;
    at[i] = off;
    off += sizes[i];
  }
  if (out != nullptr && ws != nullptr && off <= ws_bytes) {
    char* b = reinterpret_cast<char*>(ws);
    out->counter = reinterpret_cast<int*>(b + at[0]);
    out->cq = reinterpret_cast<double*>(b + at[1]);
    out->S = reinterpret_cast<double*>(b + at[2]);
    out->part = reinterpret_cast<double*>(b + at[3]);
  }
  return off;
}

// fold rows per window a workspace of ws_bytes holds (0 if not even one row)
static size_t rows_held(size_t ws_bytes, int wp) {
  const double per_row = 8.0 + 8.0 * wp + wp / 16.0;   // growth of the layout per row: c_q, folds, partials
  const size_t fixed = long_ram_layout(nullptr, 0, wp, 0, nullptr);
  if (ws_bytes <= fixed) return 0;
  size_t rc = (size_t)((double)(ws_bytes - fixed) / per_row);
  while (rc > 0 && long_ram_layout(nullptr, 0, wp, rc + 1, nullptr) <= ws_bytes) ++rc;
  while (rc > 0 && long_ram_layout(nullptr, 0, wp, rc, nullptr) > ws_bytes) --rc;
  return rc;
}

}  // namespace
}  // namespace pp

using namespace pp;

extern "C" {

size_t pp_long_ramanujan_workspace_bytes(int32_t B, int32_t N, int32_t qmin, int32_t qmax) {
  if (B < 0 || N < 2 || qmin < 1 || qmax < qmin || qmax > N) return 0;
  const int wp = piece_windows(B);
  const size_t rows = cq_offset(qmax + 1) - cq_offset(qmin);
  size_t rc = kLrFoldBudget / (8 * ((size_t)wp + 1));
  if (rc > rows) rc = rows;
  if (rc < (size_t)qmax) rc = qmax;
  return long_ram_layout(nullptr, 0, wp, rc, nullptr);
}

int pp_long_ramanujan_norms(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t qmin, int32_t qmax,
                            const int32_t* mu, const int32_t* phi, int32_t table_qmax, double* norms, int32_t ld_norms,
                            void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (x == nullptr || norms == nullptr || B < 0 || N < 2 || ldx < 1) return fail(-1, "bad window arguments%s");
  if (qmin < 1 || qmax < qmin || qmax > N) return fail(-1, "need 1 <= qmin <= qmax <= N%s");
  if (mu == nullptr || phi == nullptr || table_qmax < qmax) return fail(-1, "mu/phi tables must cover qmax%s");
  if (ld_norms < qmax + 1) return fail(-1, "bad norms leading dimension%s");
  const int wp = piece_windows(B);
  size_t rc = workspace == nullptr ? 0 : rows_held(workspace_bytes, wp);
  if (rc < (size_t)qmax) return fail(-3, "workspace too small (see pp_long_ramanujan_workspace_bytes)%s");
  DeviceFacts f;
  if (int rc_dev = device_facts(f)) return rc_dev;
  // the folds and c_q of a chunk stay within half the L2 cache (one period always fits, whatever its size)
  size_t rc_l2 = (size_t)l2_bytes() / 2 / (8 * ((size_t)wp + 1));
  if (rc_l2 < (size_t)qmax) rc_l2 = qmax;
  if (rc > rc_l2) rc = rc_l2;
  LongRamWs w;
  long_ram_layout(workspace, workspace_bytes, wp, rc, &w);
  const size_t pc = partial_cap(rc);
  if (int rcode = prep_kernel(long_ram_dmma_kernel, kLrSmem, f)) return rcode;
  const int ctas = grid_for(f, kLrSmem, 0, 2);
  cudaStream_t st = (cudaStream_t)stream;
  for (int b0 = 0; b0 < B; b0 += wp) {
    const int nw = B - b0 < wp ? B - b0 : wp;
    const int gfull = nw / 8, nlone = nw % 8;   // pieces are multiples of 8 windows but the last
    const double* xp = x + (size_t)b0 * ldx;
    for (int qb = qmax; qb >= qmin;) {
      // chunk [qa, qb]: folds within rc rows, partial norms within pc, periods within one grid dimension
      const int nrbs = lr_blocks(qb, 1);
      size_t rows = 0;
      long long units = 0;
      int qa = qb;
      while (qa >= qmin && rows + qa <= rc && (size_t)(qb - qa + 1) * nrbs <= pc && qb - qa + 1 <= 65535) {
        rows += qa;
        units += lr_units(qa, gfull, nlone);
        --qa;
      }
      ++qa;
      const int nq = qb - qa + 1;
      long_ram_cq_kernel<<<nq, 256, 0, st>>>(qa, qb, mu, phi, w.cq);
      const long long fblocks = ((long long)qb * nw + kThreads - 1) / kThreads;
      long_ram_fold_kernel<<<dim3(fblocks < 128 ? (unsigned)fblocks : 128u, nq), kThreads, 0, st>>>(
          xp, ldx, nw, gfull, N, qa, qb, w.S, rc);
      if (int rcode = check_cuda(cudaMemsetAsync(w.counter, 0, sizeof(int), st), "cudaMemsetAsync")) return rcode;
      LongRamArgs a;
      a.S = w.S;
      a.cq = w.cq;
      a.part = w.part;
      a.counter = w.counter;
      a.rc = rc;
      a.qa = qa;
      a.qb = qb;
      a.nq = nq;
      a.nrbs = nrbs;
      a.gfull = gfull;
      a.nlone = nlone;
      a.N = N;
      a.units = units;
      long_ram_dmma_kernel<<<units < ctas ? (int)units : ctas, kThreads, kLrSmem, st>>>(a);
      long_ram_reduce_kernel<<<(nw * nq + 255) / 256, 256, 0, st>>>(w.part, nw, gfull, qa, nq, nrbs, phi,
                                                                   norms + (size_t)b0 * ld_norms, ld_norms);
      if (int rcode = check_cuda(cudaGetLastError(), "long ramanujan kernels launch")) return rcode;
      qb = qa - 1;
    }
  }
  return 0;
}

}  // extern "C"
