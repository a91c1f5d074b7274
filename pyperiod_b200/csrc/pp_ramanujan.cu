// pyperiod_b200 -- Ramanujan periodogram (pyPeriod/RamanujanPeriods.py:67-86, 124-169) on the B200.
//
// Reference, per period q: dictionary of q rows (c_q rolled by i, tiled to N), each rescaled by its
// maximum phi(q); projection  output = sum_i <x, r_i> r_i ;  norms[q] = sum_n output[n]^2.
// With S_q the residue-class fold of the window and C[i][m] = c_q((m - i) mod q) / phi(q):
//     y = C S_q,  z = C^T y,  norms[q] = sum_m cnt_q[m] z_m^2        (SURVEY.md 8a row 8)
// and since the circular autocorrelation of a Ramanujan sum is q c_q, C^T C = (q / phi^2) circ(c_q):
//     z = (q / phi(q)^2) * H S_q,   H[m][l] = c_q((l - m) mod q)      (integer matrix).
//
// Three kernels:
//   cq_kernel        the dictionary: c_q(n) = mu(q/g) phi(q) / phi(q/g), g = gcd(n, q), exact integers
//   fold_all_kernel  S_q for every q of every window of a tile (4 windows per CTA staged in shared memory)
//   ram_gemm_kernel  the dense contraction  H (q x q) * S_q (q x Bt)  on the FP64 tensor cores
//                    (mma.sync m8n8k4 f64 = DMMA) with the cnt-weighted column norms fused in the epilogue.
// H is never materialised: its fragments are generated from the q-vector c_q held in shared memory.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pyperiod_b200.h"
#include "pp_common.cuh"
#include "pp_host.cuh"

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

enum { kModeF64 = PP_RAM_FP64, kModeTf32 = PP_RAM_TF32, kModeF32Compat = PP_RAM_F32COMPAT };

// ------------------------------------------------------------------------------------------
// dictionary: c_q(n) for all q in [0, qmax], concatenated at offset cq_offset(q) = q (q - 1) / 2 (triangular layout)
// ------------------------------------------------------------------------------------------
__global__ void cq_kernel(int qmin, int qmax, const int32_t* __restrict__ mu, const int32_t* __restrict__ phi,
                          double* __restrict__ cq) {
  const int q = qmin + blockIdx.x;
  if (q > qmax) return;
  double* out = cq + cq_offset(q);
  for (int n = threadIdx.x; n < q; n += blockDim.x) out[n] = ramanujan_sum(n, q, mu, phi);
}

// ------------------------------------------------------------------------------------------
// fold of every period for a tile of windows: S[soff(q) + m * ldS + b]
// ------------------------------------------------------------------------------------------
constexpr int kFoldWin = 4;  // windows per CTA: one 32-byte sector of S per (q, m)

__host__ __device__ inline size_t s_offset(int q, int qmin, size_t ldS) {
  // rows of all periods below q: sum_{t=qmin}^{q-1} t
  return ((size_t)q * (q - 1) / 2 - (size_t)qmin * (qmin - 1) / 2) * ldS;
}

__global__ void __launch_bounds__(kThreads, 1)
fold_all_kernel(const double* __restrict__ x, int64_t ldx, int b_first, int b_count, int N, int qmin, int qmax,
                double* __restrict__ S, int ldS) {
  double* xs = reinterpret_cast<double*>(pp_smem);  // [kFoldWin][nstride]
  const int nstride = (N + 1) & ~1;
  __shared__ int counter;
  const int lane = threadIdx.x & 31;
  for (int g0 = blockIdx.x * kFoldWin; g0 < b_count; g0 += gridDim.x * kFoldWin) {
    __syncthreads();
    for (int w = 0; w < kFoldWin; ++w) {
      const bool live = g0 + w < b_count;
      const double* src = x + (size_t)(b_first + g0 + w) * ldx;
      for (int n = threadIdx.x; n < N; n += kThreads) xs[w * nstride + n] = live ? __ldg(src + n) : 0.0;
    }
    if (threadIdx.x == 0) counter = 0;
    __syncthreads();
    while (true) {
      int idx = 0;
      if (lane == 0) idx = atomicAdd(&counter, 1);
      idx = __shfl_sync(0xffffffffu, idx, 0);
      const int q = qmax - idx;  // large periods first
      if (q < qmin) break;
      double* out = S + s_offset(q, qmin, ldS) + g0;
      for (int m = lane; m < q; m += 32) {
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
        for (int n = m; n < N; n += q) {  // terms in increasing n, as the reference's np.dot would see them folded
          a0 += xs[n];
          a1 += xs[nstride + n];
          a2 += xs[2 * nstride + n];
          a3 += xs[3 * nstride + n];
        }
        double* o = out + (size_t)m * ldS;
        if (g0 + 3 < b_count) {
          *reinterpret_cast<double2*>(o) = make_double2(a0, a1);
          *reinterpret_cast<double2*>(o + 2) = make_double2(a2, a3);
        } else {
          o[0] = a0;
          if (g0 + 1 < b_count) o[1] = a1;
          if (g0 + 2 < b_count) o[2] = a2;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// dense contraction on the FP64 tensor cores
// ------------------------------------------------------------------------------------------
constexpr int kGemmM = 128;   // rows of H per CTA pass
constexpr int kGemmN = 64;    // windows per CTA
constexpr int kGemmK = 32;    // k-chunk staged in shared memory
constexpr int kLdB = 68;      // padded leading dimension of the staged S chunk (68 mod 16 = 4: conflict-free frags)

// grid: (ceil(Bt / 64), number of periods).  norms[(b_first + b) * ld_norms + q] = sum_m cnt_q[m] z_m^2.
__global__ void __launch_bounds__(kThreads, 2)
ram_gemm_kernel(const double* __restrict__ S, int ldS, int b_first, int b_count, int N, int qmin, int qmax,
                const double* __restrict__ cq_all, const int32_t* __restrict__ phi, double* __restrict__ norms,
                int ld_norms, double* __restrict__ zout) {
  const int q = qmax - blockIdx.y;  // big periods first
  if (q < qmin) return;
  const int b0 = blockIdx.x * kGemmN;
  if (b0 >= b_count) return;
  double* cqs = reinterpret_cast<double*>(pp_smem);              // [q]
  double* Bs0 = cqs + ((q + 1) & ~1);                              // [2][kGemmK][kLdB]: double-buffered S chunk
  double* red = Bs0 + 2 * kGemmK * kLdB;                           // [4][kGemmN]
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int wm = wid >> 1, wn = wid & 1;                           // warp tile: rows wm*32.., cols wn*32..
  const int lr = lane >> 2, lc = lane & 3;
  const double* cq = cq_all + cq_offset(q);
  for (int i = tid; i < q; i += kThreads) cqs[i] = cq[i];
  const double* Sq = S + s_offset(q, qmin, ldS) + b0;
  const int Mrows = N / q, r0 = N - Mrows * q;

  double colacc[4][2];
#pragma unroll
  for (int j = 0; j < 4; ++j) colacc[j][0] = colacc[j][1] = 0.0;

  for (int m0 = 0; m0 < q; m0 += kGemmM) {
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    // stage S_q[l0 .. l0+31][b0 .. b0+63] with cp.async (rows past q and windows past the tile are zero-filled);
    // the copy of chunk l0 + 32 is in flight while chunk l0 feeds the tensor cores
    auto stage = [&](double* dst, int l0) {
      for (int idx = tid; idx < kGemmK * kGemmN / 2; idx += kThreads) {
        const int kk = idx >> 5, n = (idx & 31) * 2;
        int bytes = 0;
        if (l0 + kk < q) bytes = min(max(b_count - (b0 + n), 0), 2) * 8;
        const double* src = bytes ? Sq + (size_t)(l0 + kk) * ldS + n : Sq;
        cp_async_16(dst + kk * kLdB + n, src, bytes);
      }
      cp_async_commit();
    };
    __syncthreads();  // the previous row block is done with both buffers
    stage(Bs0, 0);
    int buf = 0;
    for (int l0 = 0; l0 < q; l0 += kGemmK, buf ^= 1) {
      const double* Bs = Bs0 + buf * (kGemmK * kLdB);
      if (l0 + kGemmK < q) {
        stage(Bs0 + (buf ^ 1) * (kGemmK * kLdB), l0 + kGemmK);
        cp_async_wait<1>();
      } else {
        cp_async_wait<0>();
      }
      __syncthreads();
#pragma unroll
      for (int k4 = 0; k4 < kGemmK / 4; ++k4) {
        const int l = l0 + k4 * 4 + lc;
        double bf[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) bf[j] = Bs[(k4 * 4 + lc) * kLdB + wn * 32 + j * 8 + lr];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int m = m0 + wm * 32 + i * 8 + lr;
          double a = 0.0;
          if (m < q && l < q) {
            int d = l - m;
            if (d < 0) d += q;
            a = cqs[d];
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) dmma_m8n8k4(acc[i][j], a, bf[j]);
        }
      }
      __syncthreads();  // everyone is done with this buffer before the next iteration restages it
    }
    // float32-compat mode: the products t = H S_q themselves are kept (same layout as S) for ram_compat_kernel
    if (zout != nullptr) {
      double* Zq = zout + s_offset(q, qmin, ldS) + b0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int m = m0 + wm * 32 + i * 8 + lr;
        if (m < q) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int col = wn * 32 + j * 8 + 2 * lc;
            if (b0 + col < b_count) Zq[(size_t)m * ldS + col] = acc[i][j][0];
            if (b0 + col + 1 < b_count) Zq[(size_t)m * ldS + col + 1] = acc[i][j][1];
          }
        }
      }
    }
    // epilogue of this row block: cnt-weighted squares, accumulated per column
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + wm * 32 + i * 8 + lr;
      const double cnt = (m < q) ? (double)(Mrows + (m < r0 ? 1 : 0)) : 0.0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        colacc[j][0] = fma(cnt * acc[i][j][0], acc[i][j][0], colacc[j][0]);
        colacc[j][1] = fma(cnt * acc[i][j][1], acc[i][j][1], colacc[j][1]);
      }
    }
  }
  // reduce over the 8 row-lanes of a column pair, then over the 4 row-warps (fixed order)
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      double v = colacc[j][e];
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      colacc[j][e] = v;
    }
  __syncthreads();
  if (lr == 0) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      red[wm * kGemmN + wn * 32 + j * 8 + 2 * lc] = colacc[j][0];
      red[wm * kGemmN + wn * 32 + j * 8 + 2 * lc + 1] = colacc[j][1];
    }
  }
  __syncthreads();
  if (tid < kGemmN && b0 + tid < b_count) {
    const double ph = (double)phi[q];
    const double scale = (double)q / (ph * ph);  // C^T C = (q / phi^2) circ(c_q)
    const double t = ((red[tid] + red[kGemmN + tid]) + red[2 * kGemmN + tid]) + red[3 * kGemmN + tid];
    norms[(size_t)(b_first + b0 + tid) * ld_norms + q] = scale * scale * t;
  }
}

// ------------------------------------------------------------------------------------------
// Fused periodogram (the default fp64 path): fold and contraction in ONE kernel, the folds never leave the SM.
//
// Work unit = (period q, 8 windows).  The CTA folds the 8 windows at q straight from global memory (the windows
// of a group stay in L2 while every q passes over them) into shared memory, S[l][w] (q x 8 doubles, <= 88 KB at
// q = 1365), and contracts it with the circulant H[m][l] = c_q((l - m) mod q) on the FP64 tensor cores.  HBM
// traffic is the window itself (N * 8 bytes) plus one norm per period; the 7.5 MB of folds per window that the
// two-kernel form wrote and re-read are gone, and so is the 15 GB fold buffer.
//
//  * Two CTAs per SM: the fold of a unit is a chain of L2 round trips (latency bound), the contraction is
//    tensor-pipe bound; the co-resident CTA's contraction hides the other one's fold.
//  * 8-row fragments of H are dealt to the 8 warps round-robin (fragment f -> warp f mod 8), up to eight fragments
//    per warp pass: the tensor-core work of a unit is balanced to one fragment whatever q is (a 128-row block
//    tiling wastes up to 127 rows of every period).  The pass is compiled for every fragment count 1..8, so the
//    inner loop carries no predicates.
//  * A lane's H element for k-step k of a 32-row chunk is cq2[d + 4 k] with ONE running index d per fragment
//    (cq2 = c_q tabulated over [0, q + 32): no wrap inside a chunk): an LDS with an immediate offset.
//  * S rows are 8 doubles: the B fragment (4 rows x 8 windows) is 256 contiguous bytes, the minimum two wavefronts.
// ------------------------------------------------------------------------------------------
constexpr int kFusedWin = 8;       // windows per unit (one 8-column B fragment)
constexpr int kFusedFrags = 8;     // 8-row fragments of H per warp pass

struct FusedPlan {
  int qmax;
  __host__ __device__ int srows() const { return (qmax + 31) & ~31; }
  __host__ __device__ size_t off_cq2() const { return (size_t)srows() * kFusedWin * 8; }
  __host__ __device__ size_t off_red() const { return off_cq2() + (size_t)((qmax + 32 + 1) & ~1) * 8; }
  __host__ __device__ size_t bytes() const { return off_red() + (size_t)kWarps * kFusedWin * 8 + 16; }
};

// One warp pass: NFR fragments (rows 8 (frag0 + 8 i) .. + 7, i < NFR) against all q rows of S.
template <int NFR>
__device__ __forceinline__ void fused_pass(const double* __restrict__ Ssm, const double* __restrict__ cq2, int q,
                                           int frag0, int Mrows, int r0, double (&colacc)[2]) {
  const int lane = threadIdx.x & 31, lr = lane >> 2, lc = lane & 3;
  // running index of this lane's H element per fragment: d = (l - m) mod q at l = lc
  int d[NFR];
#pragma unroll
  for (int i = 0; i < NFR; ++i) {
    const int m = 8 * (frag0 + 8 * i) + lr;   // fragments of this warp are 8 apart
    int v = lc + q - m;                       // in (0, q + 3] for m < q
    if (v >= q) v -= q;
    d[i] = m < q ? v : 0;                     // rows past q (last fragment): any finite table entry, weight 0 below
  }
  double acc[NFR][2];
#pragma unroll
  for (int i = 0; i < NFR; ++i) acc[i][0] = acc[i][1] = 0.0;
  const double* bptr = Ssm + lc * kFusedWin + lr;
  for (int l0 = 0; l0 < q; l0 += 32) {
#pragma unroll
    for (int k4 = 0; k4 < 8; ++k4) {
      const double b = bptr[(l0 + 4 * k4) * kFusedWin];
#pragma unroll
      for (int i = 0; i < NFR; ++i) dmma_m8n8k4(acc[i], cq2[d[i] + 4 * k4], b);
    }
#pragma unroll
    for (int i = 0; i < NFR; ++i) {
      d[i] += 32;
      if (d[i] >= q) {
        d[i] -= q;
        if (d[i] >= q) d[i] %= q;   // q < 32 only
      }
    }
  }
#pragma unroll
  for (int i = 0; i < NFR; ++i) {
    const int m = 8 * (frag0 + 8 * i) + lr;
    const double cnt = m < q ? (double)(Mrows + (m < r0 ? 1 : 0)) : 0.0;
    colacc[0] = fma(cnt * acc[i][0], acc[i][0], colacc[0]);
    colacc[1] = fma(cnt * acc[i][1], acc[i][1], colacc[1]);
  }
}

// persistent grid (two CTAs per SM); units handed out by a global counter: window groups outermost (a group's
// windows stay in L2), periods descending inside a group (long units first), 8-window tiles innermost.
__global__ void __launch_bounds__(kThreads, 2)
ram_fused_kernel(const double* __restrict__ x, int64_t ldx, int B, int N, int qmin, int qmax, int group_windows,
                 const double* __restrict__ cq_all, const int32_t* __restrict__ phi, double* __restrict__ norms,
                 int ld_norms, int* __restrict__ next_unit) {
  FusedPlan pl;
  pl.qmax = qmax;
  double* Ssm = reinterpret_cast<double*>(pp_smem);
  double* cq2 = reinterpret_cast<double*>(pp_smem + pl.off_cq2());
  double* red = reinterpret_cast<double*>(pp_smem + pl.off_red());
  int* unit_slot = reinterpret_cast<int*>(red + kWarps * kFusedWin);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nq = qmax - qmin + 1;
  const int tiles_per_group = group_windows / kFusedWin;
  const int ngroups = (B + group_windows - 1) / group_windows;
  const long long per_group = (long long)nq * tiles_per_group;
  const long long nunits = per_group * ngroups;
  int q_tab = 0;   // period whose table is in cq2
  for (;;) {
    if (tid == 0) *unit_slot = atomicAdd(next_unit, 1);
    __syncthreads();   // also: every warp is done with S, cq2 and red of the previous unit
    const long long u = *unit_slot;
    if (u >= nunits) break;
    const int grp = (int)(u / per_group);
    const int rem = (int)(u - (long long)grp * per_group);
    const int q = qmax - rem / tiles_per_group;
    const int w0 = grp * group_windows + (rem % tiles_per_group) * kFusedWin;
    if (w0 >= B) {           // tail of the last group (uniform over the CTA)
      __syncthreads();       // everyone has read the unit before thread 0 draws the next one
      continue;
    }
    const int Mrows = N / q, r0 = N - Mrows * q;
    if (q != q_tab) {
      const double* cq = cq_all + cq_offset(q);
      for (int i = tid; i < q + 32; i += kThreads) cq2[i] = cq[i >= q ? (i - q) % q : i];
      q_tab = q;
    }
    // ---- fold: S[m][w] = sum_j x[w][j q + m].  A warp step covers 8 residues x 8 windows (64 contiguous bytes per
    //      window, two windows per lane); two partial sums per chain (rows j mod 2) keep four loads of a lane in
    //      flight at a time and meet in a fixed order.
    {
      const int mi = lane & 7, wi = lane >> 3;
      const int nmb = (q + 7) >> 3;
      for (int mb = wid; mb < nmb; mb += kWarps) {
        const int m = 8 * mb + mi;
        double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0;
        if (m < q) {
          const bool la = w0 + wi < B, lb = w0 + wi + 4 < B;
          const double* pa = x + (size_t)(la ? w0 + wi : w0) * ldx + m;
          const double* pb = x + (size_t)(lb ? w0 + wi + 4 : w0) * ldx + m;
          const int terms = Mrows + (m < r0 ? 1 : 0);
          int j = 0;
          for (; j + 2 <= terms; j += 2) {
            a0 += __ldg(pa + (size_t)j * q);
            a1 += __ldg(pa + (size_t)(j + 1) * q);
            b0 += __ldg(pb + (size_t)j * q);
            b1 += __ldg(pb + (size_t)(j + 1) * q);
          }
          if (j < terms) {
            a0 += __ldg(pa + (size_t)j * q);
            b0 += __ldg(pb + (size_t)j * q);
          }
          Ssm[m * kFusedWin + wi] = la ? a0 + a1 : 0.0;
          Ssm[m * kFusedWin + wi + 4] = lb ? b0 + b1 : 0.0;
        }
      }
      // rows q .. round-up to the k-chunk: zero (their H elements are finite table entries)
      const int qr = (q + 31) & ~31;
      for (int i = q * kFusedWin + tid; i < qr * kFusedWin; i += kThreads) Ssm[i] = 0.0;
    }
    __syncthreads();
    // ---- contraction: warp `wid` owns fragments wid, wid + 8, ... (8 rows each), up to eight per pass
    double colacc[2] = {0.0, 0.0};
    const int nfrag = (q + 7) >> 3;
    for (int f0 = wid; f0 < nfrag; f0 += 8 * kFusedFrags) {
      const int nfr = min(kFusedFrags, (nfrag - f0 + 7) >> 3);
      switch (nfr) {
        case 8: fused_pass<8>(Ssm, cq2, q, f0, Mrows, r0, colacc); break;
        case 7: fused_pass<7>(Ssm, cq2, q, f0, Mrows, r0, colacc); break;
        case 6: fused_pass<6>(Ssm, cq2, q, f0, Mrows, r0, colacc); break;
        case 5: fused_pass<5>(Ssm, cq2, q, f0, Mrows, r0, colacc); break;
        case 4: fused_pass<4>(Ssm, cq2, q, f0, Mrows, r0, colacc); break;
        case 3: fused_pass<3>(Ssm, cq2, q, f0, Mrows, r0, colacc); break;
        case 2: fused_pass<2>(Ssm, cq2, q, f0, Mrows, r0, colacc); break;
        default: fused_pass<1>(Ssm, cq2, q, f0, Mrows, r0, colacc); break;
      }
    }
    // column sums: over the 8 row-lanes of a fragment, then over the warps in a fixed order
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      double v = colacc[e];
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      colacc[e] = v;
    }
    if (lane < 4) {
      red[wid * kFusedWin + 2 * lane] = colacc[0];
      red[wid * kFusedWin + 2 * lane + 1] = colacc[1];
    }
    __syncthreads();
    if (tid < kFusedWin && w0 + tid < B) {
      const double ph = (double)phi[q];
      const double scale = (double)q / (ph * ph);   // C^T C = (q / phi^2) circ(c_q)
      double t = 0.0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) t += red[w * kFusedWin + tid];
      norms[(size_t)(w0 + tid) * ld_norms + q] = scale * scale * t;
    }
  }
}

// ------------------------------------------------------------------------------------------
// TF32 option: the same contraction on the 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulator in
// tensor memory).  c_q(n) is an integer with |c_q| <= phi(q) < 2^11, exact in TF32; the fold sums are split into
// hi + lo TF32 parts, both accumulated into the SAME tensor-memory tile (two MMAs per k-step), which leaves ~2^-21
// relative error per product and the fp32 accumulation of q terms: norms agree with the fp64 path to ~1e-5.
//
// Orientation: D[w][m] = sum_k A[w][k] B[m][k] with A[w][k] = S_q[k] of window w (UMMA M = 128 windows, one
// tensor-memory lane per window) and B[m][k] = c_q((k - m) mod q) (UMMA N = up to 256 output residues).  Each
// epilogue thread owns one window (one TMEM lane) and accumulates cnt_m * z_m^2 over its columns: no cross-lane
// reduction.  Both operands are K-major tiles of 32 tf32 (one 128-byte row per window / residue) in the canonical
// SWIZZLE_128B layout, written by the CTA's own threads (the circulant is generated from c_q, the fold sums are
// converted from fp64) and handed to the tensor core through fence.proxy.async; two stages, so the tiles of
// k-block i+1 are built while the MMAs of k-block i run (tcgen05.commit -> mbarrier releases a stage).
// ------------------------------------------------------------------------------------------
constexpr int kUW = 128;          // windows per work unit (UMMA M)
constexpr int kUN = 512;          // output residues per accumulator tile: ALL 512 tensor-memory columns, two UMMAs of
                                  // N <= 256 per k-step -- the kernel is bound by fetching the folds (once per tile), so
                                  // a tile twice as wide halves that traffic
constexpr int kUNh = 256;         // UMMA N of one half
constexpr int kUK = 32;           // tf32 per k-block: one 128-byte swizzle row
constexpr int kUStageBytes = (2 * kUW + kUN) * 128;   // A_hi | A_lo | B
constexpr int kUStages = 2;

__device__ __forceinline__ uint32_t to_tf32(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return r;
}
// byte offset of 16-byte chunk c of row r in a K-major SWIZZLE_128B tile (8-row groups of 1024 bytes)
__device__ __forceinline__ uint32_t sw128_off(int r, int c) {
  return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4));
}
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 [0,14), leading byte offset >> 4
// [16,30) (1: unused for swizzled K-major), stride byte offset >> 4 [32,46) (1024 bytes between 8-row groups),
// version 1 [46,48), layout SWIZZLE_128B = 2 [61,64)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32 [4,6), A = B = TF32 (2) [7,10) [10,13), both K-major,
// N >> 3 [17,23), M >> 4 [24,29)
__device__ __forceinline__ uint32_t umma_idesc_tf32(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared-memory plan of the tcgen05 kernel (bytes from a 1024-aligned base)
struct UmmaPlan {
  int qpad;
  __host__ __device__ size_t off_cq() const { return (size_t)kUStages * kUStageBytes; }
  __host__ __device__ size_t off_red() const { return off_cq() + (size_t)qpad * 4; }
  __host__ __device__ size_t off_bar() const { return off_red() + (size_t)kUW * 8; }
  __host__ __device__ size_t bytes() const { return off_bar() + 64 + 1024; }   // + slack for the 1024-byte alignment
};

// persistent grid; work unit u = (period, 128-window tile), big periods first, handed out by a global counter.
// S[soff(q) + k * ldS + w] = fold sum of window w at residue k (fold_all_kernel).
__global__ void __launch_bounds__(kThreads, 1)
ram_umma_tf32_kernel(const double* __restrict__ S, int ldS, int b_first, int b_count, int N, int qmin, int qmax,
                     const double* __restrict__ cq_all, const int32_t* __restrict__ phi, double* __restrict__ norms,
                     int ld_norms, int* __restrict__ next_unit) {
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const uint32_t base_u32 = (smem_u32(pp_smem) + 1023u) & ~1023u;
  unsigned char* base = pp_smem + (base_u32 - smem_u32(pp_smem));
  UmmaPlan pl;
  pl.qpad = (qmax + 3 + 31) & ~31;
  float* cqs = reinterpret_cast<float*>(base + pl.off_cq());
  double* red = reinterpret_cast<double*>(base + pl.off_red());
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + pl.off_bar());   // [0], [1]: stage free; [2]: accumulator ready
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);
  int* unit_slot = reinterpret_cast<int*>(tmem_slot + 1);

  if (tid == 0) {
    mbar_init(bars + 0, 1);
    mbar_init(bars + 1, 1);
    mbar_init(bars + 2, 1);
  }
  if (wid == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kUN));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;

  const int ntiles_w = (b_count + kUW - 1) / kUW;
  const int nunits = (qmax - qmin + 1) * ntiles_w;
  uint32_t phase0 = 0, phase1 = 0, phase_acc = 0;   // mbarrier parities (uniform over the CTA)
  bool pend0 = false, pend1 = false;                 // a commit on the stage barrier has not been waited for yet

  for (;;) {
    if (tid == 0) *unit_slot = atomicAdd(next_unit, 1);
    __syncthreads();
    const int u = *unit_slot;
    if (u >= nunits) break;
    const int q = qmax - u / ntiles_w;
    const int w0 = (u % ntiles_w) * kUW;
    const double* cq = cq_all + cq_offset(q);
    for (int i = tid; i < q; i += kThreads) cqs[i] = (float)cq[i];
    const double* Sq = S + s_offset(q, qmin, ldS) + w0;
    const int wlive = min(kUW, b_count - w0);
    const int Mrows = N / q, r0 = N - Mrows * q;
    const int nkb = (q + kUK - 1) / kUK;
    double wacc = 0.0;   // this thread's window: sum of cnt_m z_m^2 over its half of the columns
    __syncthreads();

    for (int m0 = 0; m0 < q; m0 += kUN) {
      const int nt = min(kUN, (q - m0 + 15) & ~15);       // columns of this accumulator tile (multiple of 16)
      const int nt0 = min(nt, kUNh), nt1 = nt - nt0;      // UMMA N of the two halves (nt1 may be 0)
      const uint32_t idesc0 = umma_idesc_tf32(kUW, nt0), idesc1 = umma_idesc_tf32(kUW, nt1 > 0 ? nt1 : 16);
      for (int kb = 0; kb < nkb; ++kb) {
        const int st = kb & 1;
        unsigned char* stage = base + (size_t)st * kUStageBytes;
        // the MMAs that read this stage two k-blocks ago must be done before it is rewritten
        if (st == 0 ? pend0 : pend1) {
          mbar_wait(bars + st, st == 0 ? phase0 : phase1);
          if (st == 0) { phase0 ^= 1u; pend0 = false; } else { phase1 ^= 1u; pend1 = false; }
        }
        const int k0 = kb * kUK;
        // ---- A tiles: fold sums of 128 windows x 32 residues, fp64 -> tf32 hi + lo.  One thread = one window row and
        //      one 16-byte chunk (4 consecutive residues) per step; reads are coalesced over the windows.
        for (int idx = tid; idx < kUW * 8; idx += kThreads) {
          const int w = idx & (kUW - 1), c = idx >> 7;
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int k = k0 + 4 * c + e;
            double v = 0.0;
            if (k < q && w < wlive) v = Sq[(size_t)k * ldS + w];
            const uint32_t h = to_tf32((float)v);
            hi[e] = h;
            lo[e] = to_tf32((float)(v - (double)__uint_as_float(h)));
          }
          const uint32_t off = sw128_off(w, c);
          *reinterpret_cast<uint4*>(stage + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4*>(stage + kUW * 128 + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
        // ---- B tile: the circulant, B[m][k] = c_q((k - m) mod q), generated from c_q
        for (int idx = tid; idx < nt * 8; idx += kThreads) {
          const int r = idx >> 3, c = idx & 7;
          const int m = m0 + r;
          float v[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int k = k0 + 4 * c + e;
            float x = 0.f;
            if (m < q && k < q) {
              int d = k - m;
              if (d < 0) d += q;
              x = cqs[d];
            }
            v[e] = x;
          }
          *reinterpret_cast<float4*>(stage + 2 * kUW * 128 + sw128_off(r, c)) = make_float4(v[0], v[1], v[2], v[3]);
        }
        fence_proxy_async();          // generic-proxy writes -> visible to the tensor core's async-proxy reads
        __syncthreads();
        if (tid == 0) {
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t sa = base_u32 + (uint32_t)st * kUStageBytes;
          const uint64_t a_hi = umma_desc_sw128(sa), a_lo = umma_desc_sw128(sa + kUW * 128),
                         bd = umma_desc_sw128(sa + 2 * kUW * 128);
#pragma unroll
          const uint64_t bd1 = umma_desc_sw128(sa + 2 * kUW * 128 + kUNh * 128);   // rows 256.. of the B tile
          for (int k = 0; k < kUK / 8; ++k) {   // UMMA K = 8 tf32 = 32 bytes: advance the start address by 2 (x16 B)
            const uint32_t accum = (kb > 0 || k > 0) ? 1u : 0u;
            umma_tf32(tmem, a_hi + 2 * k, bd + 2 * k, idesc0, accum);
            umma_tf32(tmem, a_lo + 2 * k, bd + 2 * k, idesc0, 1u);
            if (nt1 > 0) {                      // second half: tensor-memory columns 256 ..
              umma_tf32(tmem + kUNh, a_hi + 2 * k, bd1 + 2 * k, idesc1, accum);
              umma_tf32(tmem + kUNh, a_lo + 2 * k, bd1 + 2 * k, idesc1, 1u);
            }
          }
          umma_commit(bars + st);                       // frees this stage when the MMAs above have read it
          if (kb == nkb - 1) umma_commit(bars + 2);     // ... and the accumulator tile is complete
        }
        if (st == 0) pend0 = true; else pend1 = true;
      }
      // ---- epilogue of this accumulator tile: lane = window, columns = output residues m0 .. m0 + nt
      mbar_wait(bars + 2, phase_acc);
      phase_acc ^= 1u;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      {
        const int half = wid >> 2;                         // warps 0-3: columns [0, 256), warps 4-7: [256, 512)
        const uint32_t lane_base = (uint32_t)(32 * (wid & 3)) << 16;
        for (int c0 = half * kUNh; c0 < min(nt, half * kUNh + kUNh); c0 += 32) {
          uint32_t r[32];
          tmem_ld_x32(tmem + lane_base + (uint32_t)c0, r);
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int m = m0 + c0 + j;
            if (m < q) {
              const double z = (double)__uint_as_float(r[j]);
              wacc = fma((double)(Mrows + (m < r0 ? 1 : 0)) * z, z, wacc);
            }
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();   // every warp has read the tile before the next one overwrites it
    }
    // ---- norms of this unit: the two column halves of a window meet in shared memory
    const int w = 32 * (wid & 3) + lane;
    if (wid >= 4) red[w] = wacc;
    __syncthreads();
    if (wid < 4 && w < wlive) {
      const double ph = (double)phi[q];
      const double scale = (double)q / (ph * ph);
      norms[(size_t)(b_first + w0 + w) * ld_norms + q] = scale * scale * (wacc + red[w]);
    }
    __syncthreads();
  }
  // drain: nothing asynchronous may still reference this CTA's shared memory or tensor memory
  if (pend0) mbar_wait(bars + 0, phase0);
  if (pend1) mbar_wait(bars + 1, phase1);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (wid == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kUN));
}

// ------------------------------------------------------------------------------------------
// float32-compat mode: the reference's OWN numbers.  RamanujanPeriods.project stores every projected row in a
// float32 array (RamanujanPeriods.py:127-130), find_periods sums the q rows in float32 (np.sum over axis 0:
// sequential in the row index) and then sums the squares of the N float32 samples with numpy's pairwise summation
// (:77-78).  That rounding noise (1e-7 .. 2e-6 relative) is the distance between the reference and the fp64 value
// of the same formula; this kernel reproduces it operation by operation:
//   y_i      = <x, r_i>                       fp64  (t_i / phi(q), t = H S_q from the DMMA kernel)
//   p_i[m]   = float32(y_i * r_i[m])          r_i[m] = c_q((m - i) mod q) / phi(q), fp64 product rounded once
//   out[m]   = ((p_0[m] + p_1[m]) + p_2[m]) + ...   float32, in row order   (out[n] depends on n mod q only)
//   norms[q] = pairwise_float32(out[n mod q]^2, n < N)   numpy's 8-way unrolled blocks of <= 128, split in halves
// What cannot be reproduced is the 1e-13 noise of the reference's sum of complex exponentials in Cq (:142-144): it
// moves a float32 rounding once in ~1e6 products.
// ------------------------------------------------------------------------------------------
constexpr int kCompatWin = 4;   // windows per CTA
constexpr int kCompatLeafCap = 512;   // leaves of the pairwise summation (N <= 32768)

// leaves of numpy's pairwise summation of n elements (blocks of <= 128; halves rounded down to a multiple of 8)
__device__ int pairwise_leaves(int n, int* off, int* len, int cap) {
  int stack_o[32], stack_n[32], sp = 0, cnt = 0;
  stack_o[0] = 0;
  stack_n[0] = n;
  sp = 1;
  while (sp > 0) {
    --sp;
    const int o = stack_o[sp], m = stack_n[sp];
    if (m <= 128) {
      if (cnt < cap) {
        off[cnt] = o;
        len[cnt] = m;
      }
      ++cnt;
    } else {
      int n2 = m / 2;
      n2 -= n2 % 8;
      stack_o[sp] = o + n2;   // right half is pushed first: the left half is visited first (in order)
      stack_n[sp] = m - n2;
      ++sp;
      stack_o[sp] = o;
      stack_n[sp] = n2;
      ++sp;
    }
  }
  return cnt;
}

// recombination of the leaf sums in recursion order: result = sum(left) + sum(right), float32
__device__ float pairwise_combine(int n, const float* leaf, int& next) {
  if (n <= 128) return leaf[next++];
  int n2 = n / 2;
  n2 -= n2 % 8;
  const float a = pairwise_combine(n2, leaf, next);
  const float b = pairwise_combine(n - n2, leaf, next);
  return __fadd_rn(a, b);
}

__global__ void __launch_bounds__(kThreads, 2)
ram_compat_kernel(const double* __restrict__ Z, int ldS, int b_first, int b_count, int N, int qmin, int qmax,
                  const double* __restrict__ cq_all, const int32_t* __restrict__ phi, double* __restrict__ norms,
                  int ld_norms) {
  const int q = qmax - blockIdx.y;
  if (q < qmin) return;
  const int w0 = blockIdx.x * kCompatWin;
  if (w0 >= b_count) return;
  const int qe = (q + 1) & ~1;
  double* rtab = reinterpret_cast<double*>(pp_smem);          // [q]  c_q(d) / phi(q)
  double* y = rtab + qe;                                        // [kCompatWin][q]
  float* o32 = reinterpret_cast<float*>(y + kCompatWin * qe);   // [kCompatWin][q]
  float* leaf = o32 + kCompatWin * qe;                          // [kCompatWin][nleaf_cap]
  constexpr int kLeafCap = kCompatLeafCap;
  int* loff = reinterpret_cast<int*>(leaf + kCompatWin * kLeafCap);
  int* llen = loff + kLeafCap;
  __shared__ int s_nleaf;
  const int tid = threadIdx.x;
  const double ph = (double)phi[q];
  const double* cq = cq_all + cq_offset(q);
  const double* Zq = Z + s_offset(q, qmin, ldS) + w0;
  for (int i = tid; i < q; i += kThreads) rtab[i] = cq[i] / ph;          // row / max(row): c_q / phi(q)
  for (int idx = tid; idx < kCompatWin * q; idx += kThreads) {
    const int w = idx / q, i = idx - w * q;
    y[w * qe + i] = (w0 + w < b_count) ? Zq[(size_t)i * ldS + w] / ph : 0.0;   // <x, r_i> = t_i / phi(q)
  }
  if (tid == 0) s_nleaf = pairwise_leaves(N, loff, llen, kLeafCap);
  __syncthreads();
  // out[m] = sequential float32 sum over the rows i of float32(y_i * r_i[m])
  for (int idx = tid; idx < kCompatWin * q; idx += kThreads) {
    const int w = idx / q, m = idx - w * q;
    const double* yw = y + w * qe;
    int d = m;                                   // (m - i) mod q
    float acc = __double2float_rn(yw[0] * rtab[d]);
    for (int i = 1; i < q; ++i) {
      d = d == 0 ? q - 1 : d - 1;
      acc = __fadd_rn(acc, __double2float_rn(yw[i] * rtab[d]));
    }
    o32[w * qe + m] = acc;
  }
  __syncthreads();
  // squares, pairwise: every leaf keeps numpy's 8 strided partial sums; one thread per (window, leaf, lane-of-8)
  const int nleaf = min(s_nleaf, kLeafCap);
  for (int idx = tid; idx < kCompatWin * nleaf * 8; idx += kThreads) {
    const int j = idx & 7, l = (idx >> 3) % nleaf, w = idx / (8 * nleaf);
    const float* ow = o32 + w * qe;
    const int o = loff[l], n = llen[l];
    float r = 0.f;
    if (n >= 8) {
      int pos = (o + j) % q;
      const int step = 8 % q;
      float v = ow[pos];
      r = __fmul_rn(v, v);
      for (int i = 8; i < n - (n % 8); i += 8) {
        pos += step;
        if (pos >= q) pos -= q;
        v = ow[pos];
        r = __fadd_rn(r, __fmul_rn(v, v));
      }
    }
    // the 8 partial sums of a leaf meet through shuffles: lanes j .. j+7 of the same leaf are adjacent
    const float r1 = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 1));      // (r0+r1), (r2+r3), ...
    const float r2 = __fadd_rn(r1, __shfl_xor_sync(0xffffffffu, r1, 2));    // ((r0+r1)+(r2+r3)), ...
    float res = __fadd_rn(r2, __shfl_xor_sync(0xffffffffu, r2, 4));
    if (j == 0) {
      if (n < 8) {
        res = 0.f;
        for (int i = 0; i < n; ++i) {
          const float v = ow[(o + i) % q];
          res = __fadd_rn(res, __fmul_rn(v, v));
        }
      } else {
        for (int i = n - (n % 8); i < n; ++i) {
          const float v = ow[(o + i) % q];
          res = __fadd_rn(res, __fmul_rn(v, v));
        }
      }
      leaf[w * kLeafCap + l] = res;
    }
  }
  __syncthreads();
  if (tid < kCompatWin && w0 + tid < b_count) {
    int next = 0;
    const float total = __fadd_rn(0.f, pairwise_combine(N, leaf + tid * kLeafCap, next));
    norms[(size_t)(b_first + w0 + tid) * ld_norms + q] = (double)total;
  }
}

// periods whose norm exceeds thresh * |max norm|, ascending (RamanujanPeriods.py:97-101); one warp per window
__global__ void select_kernel(const double* __restrict__ norms, int B, int ld_norms, int qlen, double thresh, int kmax,
                              int32_t* __restrict__ periods, int32_t* __restrict__ nper) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  const double* nr = norms + (size_t)b * ld_norms;
  double mx = -1.0 / 0.0;
  for (int q = lane; q < qlen; q += 32) mx = fmax(mx, nr[q]);
  mx = warp_max(mx);
  const double den = fabs(mx);
  int count = 0;
  for (int q0 = 0; q0 < qlen; q0 += 32) {
    const int q = q0 + lane;
    const bool hit = q < qlen && (nr[q] / den > thresh);
    const unsigned mask = __ballot_sync(0xffffffffu, hit);
    if (hit) {
      const int pos = count + __popc(mask & ((1u << lane) - 1u));
      if (pos < kmax) periods[(size_t)b * kmax + pos] = q;
    }
    count += __popc(mask);
  }
  if (lane == 0) nper[b] = count;
}

}  // namespace pp

using namespace pp;

extern "C" {

// mode: PP_RAM_FP64 (fused kernel: the dictionary table and a counter), PP_RAM_TF32 (folds of one tile),
// PP_RAM_F32COMPAT (folds and products of one tile)
size_t pp_ramanujan_workspace_bytes(int32_t N, int32_t qmin, int32_t qmax, int32_t tile_windows, int32_t mode) {
  (void)N;
  const size_t ldS = ((size_t)tile_windows + 3) & ~(size_t)3;
  const size_t rows = (size_t)qmax * (qmax + 1) / 2 - (size_t)qmin * (qmin - 1) / 2;
  size_t bytes = 4096 + 256 + (cq_offset(qmax + 1) + 2) * 8;
  if (mode == kModeTf32 || mode == kModeF32Compat) bytes += rows * ldS * 8;
  if (mode == kModeF32Compat) bytes += 256 + rows * ldS * 8;
  return bytes;
}

// Shared memory per block of every kernel a mode launches.  The launch below and pp_ramanujan_fits_on_chip both
// evaluate this plan, so the library's choice between the on-chip and the global-memory periodogram is the launch's.
struct RamanujanPlan {
  size_t fused, fold, gemm, umma, compat;
};
static RamanujanPlan ramanujan_plan(int N, int qmax) {
  RamanujanPlan p;
  FusedPlan fpl;
  fpl.qmax = qmax;
  p.fused = fpl.bytes();
  p.fold = (size_t)kFoldWin * ((N + 1) & ~1) * 8;
  p.gemm = (size_t)(((qmax + 1) & ~1) + 2 * kGemmK * kLdB + 4 * kGemmN) * 8;
  UmmaPlan upl;
  upl.qpad = (qmax + 3 + 31) & ~31;
  p.umma = upl.bytes();
  const size_t qe_max = (size_t)((qmax + 1) & ~1);
  p.compat = (1 + kCompatWin) * qe_max * 8 + kCompatWin * qe_max * 4 + (size_t)kCompatWin * kCompatLeafCap * 4 +
             2 * (size_t)kCompatLeafCap * 4;
  return p;
}
static bool compat_supports(int N) { return (N + 63) / 64 <= kCompatLeafCap; }
static bool ramanujan_plan_fits(const RamanujanPlan& p, int mode, int N, size_t smem) {
  if (mode == kModeF64) return p.fused <= smem;
  if (p.fold > smem || p.gemm > smem) return false;
  if (mode == kModeTf32) return p.umma <= smem;
  return compat_supports(N) && p.compat <= smem;
}

// norms[b, q] for q in [qmin, qmax] (other entries untouched; the caller zero-fills, RamanujanPeriods.py:71).
// mu / phi: device int32 tables for 0..table_qmax.  Windows are processed in tiles of `tile_windows`
// (workspace holds the folds of one tile).
static int ramanujan_norms_impl(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t qmin, int32_t qmax,
                                const int32_t* mu, const int32_t* phi, int32_t table_qmax, int32_t tile_windows,
                                double* norms, int32_t ld_norms, void* workspace, size_t workspace_bytes, void* stream,
                                int mode) {
  const bool tf32 = mode == kModeTf32, compat = mode == kModeF32Compat;
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (x == nullptr || norms == nullptr || B < 0 || N < 2 || ldx < 1) return fail(-1, "bad window arguments%s");
  if (qmin < 1 || qmax < qmin || qmax > N) return fail(-1, "need 1 <= qmin <= qmax <= N%s");
  if (mu == nullptr || phi == nullptr || table_qmax < qmax) return fail(-1, "mu/phi tables must cover qmax%s");
  if (ld_norms < qmax + 1 || tile_windows < 1) return fail(-1, "bad norms leading dimension or tile%s");
  if (B == 0) return 0;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int ldS = (tile_windows + 3) & ~3;
  const size_t rows = (size_t)qmax * (qmax + 1) / 2 - (size_t)qmin * (qmin - 1) / 2;
  size_t off = 0;
  const bool fused = mode == kModeF64;
  const RamanujanPlan plan = ramanujan_plan(N, qmax);
  double* cq = carve(workspace, workspace_bytes, off, (cq_offset(qmax + 1) + 2) * 8);
  int* next_unit = reinterpret_cast<int*>(carve(workspace, workspace_bytes, off, 256));
  double* S = fused ? nullptr : carve(workspace, workspace_bytes, off, rows * (size_t)ldS * 8);
  double* Z = compat ? carve(workspace, workspace_bytes, off, rows * (size_t)ldS * 8) : nullptr;
  if (!cq || !next_unit || (!fused && !S) || (compat && !Z))
    return fail(-3, "workspace too small (see pp_ramanujan_workspace_bytes)%s");
  cq_kernel<<<qmax - qmin + 1, 128, 0, st>>>(qmin, qmax, mu, phi, cq);
  if (fused) {
    // one launch for the whole batch; tile_windows is the L2 group (windows re-read by every period)
    if (int rc = prep_kernel(ram_fused_kernel, plan.fused, f)) return rc;
    const int group_req = tile_windows < B ? tile_windows : B;   // a small batch is one (short) group: no empty units
    const int group = (group_req + kFusedWin - 1) / kFusedWin * kFusedWin;
    const long long units = (long long)(qmax - qmin + 1) * (group / kFusedWin) * ((B + group - 1) / group);
    if (units > 0x7fffffffLL) return fail(-1, "batch too large for one launch%s");
    if (int rc = check_cuda(cudaMemsetAsync(next_unit, 0, sizeof(int), st), "cudaMemsetAsync")) return rc;
    const int ctas = grid_for(f, plan.fused, 0, 2);
    const int grid = units < ctas ? (int)units : ctas;
    ram_fused_kernel<<<grid, kThreads, plan.fused, st>>>(x, ldx, B, N, qmin, qmax, group, cq, phi, norms, ld_norms,
                                                         next_unit);
    return check_cuda(cudaGetLastError(), "ram_fused_kernel launch");
  }
  const size_t fold_smem = plan.fold, gemm_smem = plan.gemm, compat_smem = plan.compat;
  if (int rc = prep_kernel(fold_all_kernel, fold_smem, f)) return rc;
  if (int rc = prep_kernel(ram_gemm_kernel, gemm_smem, f)) return rc;
  if (tf32)
    if (int rc = prep_kernel(ram_umma_tf32_kernel, plan.umma, f)) return rc;
  if (compat) {
    if (!compat_supports(N)) return fail(-1, "float32-compat mode supports N <= 32768%s");
    if (int rc = prep_kernel(ram_compat_kernel, compat_smem, f)) return rc;
  }
  for (int b_first = 0; b_first < B; b_first += tile_windows) {
    const int b_count = (B - b_first < tile_windows) ? (B - b_first) : tile_windows;
    int fgrid = (b_count + kFoldWin - 1) / kFoldWin;
    if (fgrid > f.sm_count) fgrid = f.sm_count;
    fold_all_kernel<<<fgrid, kThreads, fold_smem, st>>>(x, ldx, b_first, b_count, N, qmin, qmax, S, ldS);
    dim3 grid((b_count + kGemmN - 1) / kGemmN, qmax - qmin + 1);
    if (tf32) {
      const int units = (qmax - qmin + 1) * ((b_count + kUW - 1) / kUW);
      if (int rc = check_cuda(cudaMemsetAsync(next_unit, 0, sizeof(int), st), "cudaMemsetAsync")) return rc;
      ram_umma_tf32_kernel<<<units < f.sm_count ? units : f.sm_count, kThreads, plan.umma, st>>>(
          S, ldS, b_first, b_count, N, qmin, qmax, cq, phi, norms, ld_norms, next_unit);
    } else {
      ram_gemm_kernel<<<grid, kThreads, gemm_smem, st>>>(S, ldS, b_first, b_count, N, qmin, qmax, cq, phi, norms,
                                                         ld_norms, Z);
      if (compat) {
        dim3 cgrid((b_count + kCompatWin - 1) / kCompatWin, qmax - qmin + 1);
        ram_compat_kernel<<<cgrid, kThreads, compat_smem, st>>>(Z, ldS, b_first, b_count, N, qmin, qmax, cq, phi, norms,
                                                                ld_norms);
      }
    }
  }
  return check_cuda(cudaGetLastError(), "ramanujan kernels launch");
}

int pp_ramanujan_norms(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t qmin, int32_t qmax,
                       const int32_t* mu, const int32_t* phi, int32_t table_qmax, int32_t tile_windows,
                       double* norms, int32_t ld_norms, void* workspace, size_t workspace_bytes, void* stream) {
  return ramanujan_norms_impl(x, ldx, B, N, qmin, qmax, mu, phi, table_qmax, tile_windows, norms, ld_norms, workspace,
                              workspace_bytes, stream, kModeF64);
}

int pp_ramanujan_norms_tf32(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t qmin, int32_t qmax,
                            const int32_t* mu, const int32_t* phi, int32_t table_qmax, int32_t tile_windows,
                            double* norms, int32_t ld_norms, void* workspace, size_t workspace_bytes, void* stream) {
  return ramanujan_norms_impl(x, ldx, B, N, qmin, qmax, mu, phi, table_qmax, tile_windows, norms, ld_norms, workspace,
                              workspace_bytes, stream, kModeTf32);
}

int pp_ramanujan_norms_f32compat(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t qmin, int32_t qmax,
                                 const int32_t* mu, const int32_t* phi, int32_t table_qmax, int32_t tile_windows,
                                 double* norms, int32_t ld_norms, void* workspace, size_t workspace_bytes,
                                 void* stream) {
  return ramanujan_norms_impl(x, ldx, B, N, qmin, qmax, mu, phi, table_qmax, tile_windows, norms, ld_norms, workspace,
                              workspace_bytes, stream, kModeF32Compat);
}

int pp_ramanujan_fits_on_chip(int32_t mode, int32_t N, int32_t qmin, int32_t qmax, int32_t smem_bytes) {
  if (mode != kModeF64 && mode != kModeTf32 && mode != kModeF32Compat) return -1;
  if (N < 2 || qmin < 1 || qmax < qmin || qmax > N || smem_bytes < 1) return -1;
  return ramanujan_plan_fits(ramanujan_plan(N, qmax), mode, N, (size_t)smem_bytes) ? 1 : 0;
}

// periods[b, 0:nper[b]] = ascending q in [0, qlen) with norms[b, q] / |max_q norms[b, q]| > thresh
// (RamanujanPeriods.py:97-101).  nper[b] may exceed kmax; only the first kmax are stored.
int pp_ramanujan_select(const double* norms, int32_t B, int32_t ld_norms, int32_t qlen, double thresh, int32_t kmax,
                        int32_t* periods, int32_t* nper, void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (!norms || !periods || !nper || B < 0 || qlen < 1 || ld_norms < qlen || kmax < 1)
    return fail(-1, "bad select arguments%s");
  if (B == 0) return 0;
  select_kernel<<<(B + 7) / 8, 256, 0, (cudaStream_t)stream>>>(norms, B, ld_norms, qlen, thresh, kmax, periods, nper);
  return check_cuda(cudaGetLastError(), "select_kernel launch");
}

}  // extern "C"
