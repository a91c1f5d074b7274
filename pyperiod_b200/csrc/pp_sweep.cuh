// pyperiod_b200 -- the period sweep: one warp per candidate period, residue sums in registers.
//
// Fold.  For period p a warp keeps S_p[r] for 32*J consecutive residues (r = ra + lane + 32 j) in
// registers and walks the rows k of the (rows x p) rectangle: every shared-memory read is 32
// consecutive doubles (conflict-free, 2 wavefronts) feeding exactly one DADD, so the sweep sits on
// the shared-memory roofline (8 B per add; SURVEY.md 8d).  Sums are sequential in n -- the order
// numpy uses -- so MAXABS metrics are bit-exact; energies agree with the reference's BLAS norm to
// a few ulp.
//
// Direct fold: two tiles per period.  With M = floor(N/p) and rr = N - M p, residues r < rr have M+1 terms
// and the others M.  Register tiles never straddle rr: tile A = [0, rr) runs M+1 rows, tile B = [rr, p)
// runs M rows (so the zero padding of the last row is never read), and the energy needs no per-lane
// count logic:  E = T/M + (1/(M+1) - 1/M) * T_A  with T the plain sum of squares.
//
// Hierarchical fold (ranking sweeps only).  Only the "top" periods q in (pmax/2, pmax] are folded
// from the window; S_p for every smaller candidate follows from S_2p[r] + S_2p[r + p].  A top
// q = g * 2^L (L <= 3) is folded at base period g with 2^L accumulator sets selected by
// (row - M0) mod 2^L (so the partial tail row always lands in set 0 and one code path covers the
// whole residue range); pairwise in-register adds give q/2 .. g, and if g is still even the chain
// goes on through a small per-warp scratch.  Tops that are 3/2 or 3/4 of an even top ride on its pass
// (3 * 2^L sets).  Sums differ from the sequential ones by rounding only.
//
// Nomination + verification.  Where the reference's result depends on bit-exact sums (MAXABS of
// best-correlation) or the ranking runs in float (optional), the hierarchical pass only nominates:
// every candidate whose error bound reaches the best one is folded sequentially in fp64 and ranked with
// the reference's rule (cta_sweep).
//
// Candidates are ranked by the squared metric (energy, or energy / p compared by cross
// multiplication); the square root and divisions are taken once, for the winner.
#pragma once

#include "pp_common.cuh"
#include "../../include/pyperiod_b200.h"

namespace pp {

enum PassMode { kPassEnergy = 0, kPassEnergyTail = 1, kPassMaxAbs = 2, kPassStore = 3 };

constexpr int kRcpTab = 256;

// Lives in shared memory (one per CTA), written by thread 0 before a sweep.
struct SweepParams {
  int N;
  int pmin, pmax;     // inclusive candidate range
  int metric;         // PP_METRIC_*
  int trunc;
  int orth;
  const int32_t* chain_off;  // device tables (orth only)
  const int32_t* chain_q;
  double* warp_scr;   // per-warp global scratch, 2*pv doubles (orth only)
  int pv;
  double sqrtN;
  double e_res;       // ||residual||^2   (IMPOSED)
  double data_norm;   // ||x||/sqrt(N)    (IMPOSED)
  double e_f32;       // >= sum x^2 of the swept signal: scale of the fp32 nomination's error bound (f32_energy_tol)
  double thresh;      // IMPOSED early-stop threshold; <0 disables first-hit mode
  const uint32_t* skip;  // bitmap of periods to ignore (M-best), nullable
  int nskip;             // number of bits set in skip (0 => the bitmap is not consulted)
  double* metric_out;    // global [pmax+1], nullable
  double* hier_scr;      // shared scratch of the hierarchical sweep: kWarps * hier_len doubles (nullable => direct)
  int hier_len;
  const double* rcp;     // shared table rcp[m] = 1.0 / m for m < kRcpTab (energy weights without a division)
  const uint2* tops;     // global: descriptors of the hierarchical tops in hand-out order (tops_kernel)
  int ntops;
  double* verify_keys;   // [pmax+1] (global or shared), nullable: lets MAXABS sweeps rank hierarchically (needs e_res = sum x^2)
  // fp32 nomination (NORM / GAMMA ranking sweeps): two float copies of the window in shared memory, xf1[n] = x[n+1],
  // so that a pair of consecutive samples can always be read with one aligned 8-byte load.  Needs verify_keys
  // and e_f32 >= sum x^2 of the swept signal.  offset 0 => fp64 hierarchical sweep.
  // (byte offsets into the kernel's dynamic shared memory, so that the loads stay LDS; 0 = none)
  int xf0_off;
  int xf1_off;
  // near-tie audit of NORM / GAMMA ranking sweeps (kSweepTieAudit): every candidate's ranking key is kept in
  // tie_keys (shared, [pmax + 1]); candidates inside the rounding bound of the best one (e_res >= sum x^2 of the
  // swept signal) are re-evaluated exactly.  tie_nom: shared bitmap, (pmax + 32) / 32 words.  canon_v / canon_u:
  // shared scratch of the exact projection, >= pmax + 2 doubles each (may alias hier_scr: dead by then).
  double* tie_keys;
  uint32_t* tie_nom;
  double* canon_v;
  double* canon_u;
};

struct SweepResult {
  double val;  // metric value of the winner (norm / gamma norm / max |S| / imposed norm)
  int p;
};

// Ranking key: energy for NORM and GAMMA (GAMMA compares energy / p by cross multiplication),
// the metric value itself for MAXABS and IMPOSED.
struct Best {
  double key;
  int p;
};

__device__ __forceinline__ bool better(int metric, double key, int p, const Best& b) {
  if (b.p == 0) return key > 0.0;
  if (metric == PP_METRIC_GAMMA) {
    const double l = key * (double)b.p, r = b.key * (double)p;
    return l > r || (l == r && p < b.p);
  }
  return key > b.key || (key == b.key && p < b.p);
}

__device__ __forceinline__ double key_to_value(int metric, double key, int p, double sqrtN) {
  if (metric == PP_METRIC_MAXABS || metric == PP_METRIC_IMPOSED) return key;
  double v = sqrt(key) / sqrtN;                            // periodic_norm, Periods.py:241
  if (metric == PP_METRIC_GAMMA) v = v / sqrt((double)p);  // Periods.py:239
  return v;
}

// loop-invariant pieces of SweepParams a warp keeps in registers while it ranks candidates
struct RankCtx {
  const uint32_t* skip;
  double* metric_out;
  double* tie_keys;
  const double* rcp;
  double sqrtN;
  int metric;
  int N;
  int pmin;
  int pmax;
};
__device__ __forceinline__ RankCtx rank_ctx(const SweepParams* sp) {
  return RankCtx{sp->nskip > 0 ? sp->skip : nullptr, sp->metric_out, sp->tie_keys, sp->rcp, sp->sqrtN, sp->metric, sp->N, sp->pmin, sp->pmax};
}
__device__ __forceinline__ void consider(const RankCtx& rc, double key, int p, Best& best) {
  const int metric = rc.metric;
  if (rc.metric_out != nullptr && (threadIdx.x & 31) == 0) rc.metric_out[p] = key_to_value(metric, key, p, rc.sqrtN);
  if (rc.tie_keys != nullptr && (threadIdx.x & 31) == 0) rc.tie_keys[p] = key;
  const uint32_t* skip = rc.skip;
  if (skip != nullptr && ((skip[p >> 5] >> (p & 31)) & 1u)) return;
  if (better(metric, key, p, best)) {
    best.key = key;
    best.p = p;
  }
}

// Per-lane variant: every lane ranks its own candidate (p == 0: none); `writer` lanes record the metric.
__device__ __forceinline__ void consider_lane(const RankCtx& rc, double key, int p, bool writer, Best& best) {
  if (p == 0) return;
  const int metric = rc.metric;
  if (rc.metric_out != nullptr && writer) rc.metric_out[p] = key_to_value(metric, key, p, rc.sqrtN);
  if (rc.tie_keys != nullptr && writer) rc.tie_keys[p] = key;
  const uint32_t* skip = rc.skip;
  if (skip != nullptr && ((skip[p >> 5] >> (p & 31)) & 1u)) return;
  if (better(metric, key, p, best)) {
    best.key = key;
    best.p = p;
  }
}

// Warp totals of K per-lane values with a transposed butterfly: K/2 + ... exchanges instead of 5 K.
// On return lane l holds the total of value l >> (5 - log2 K).  (Shuffles share the shared-memory data
// pipe the fold is bound by, so they are worth saving.)
template <int K, bool MAXOP = false>
__device__ __forceinline__ double warp_sum_multi(const double (&v)[K]) {
  static_assert(K == 1 || K == 2 || K == 4 || K == 8, "K must be 1, 2, 4 or 8");
  const int lane = threadIdx.x & 31;
  if constexpr (MAXOP) {  // same butterflies with max instead of + (MAXABS sweeps)
    auto comb = [](double a, double b) { return fmax(a, b); };
    if constexpr (K == 1) {
      return warp_max(v[0]);
    } else if constexpr (K == 2) {
      const bool hi = (lane & 16) != 0;
      double keep = comb(hi ? v[1] : v[0], __shfl_xor_sync(0xffffffffu, hi ? v[0] : v[1], 16));
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) keep = comb(keep, __shfl_xor_sync(0xffffffffu, keep, o));
      return keep;
    } else if constexpr (K == 4) {
      const bool hi = (lane & 16) != 0;
      double k0 = comb(hi ? v[2] : v[0], __shfl_xor_sync(0xffffffffu, hi ? v[0] : v[2], 16));
      double k1 = comb(hi ? v[3] : v[1], __shfl_xor_sync(0xffffffffu, hi ? v[1] : v[3], 16));
      const bool hi8 = (lane & 8) != 0;
      double keep = comb(hi8 ? k1 : k0, __shfl_xor_sync(0xffffffffu, hi8 ? k0 : k1, 8));
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) keep = comb(keep, __shfl_xor_sync(0xffffffffu, keep, o));
      return keep;
    } else {
      const bool hi = (lane & 16) != 0;
      double k4[4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        k4[i] = comb(hi ? v[4 + i] : v[i], __shfl_xor_sync(0xffffffffu, hi ? v[i] : v[4 + i], 16));
      const bool hi8 = (lane & 8) != 0;
      double k0 = comb(hi8 ? k4[2] : k4[0], __shfl_xor_sync(0xffffffffu, hi8 ? k4[0] : k4[2], 8));
      double k1 = comb(hi8 ? k4[3] : k4[1], __shfl_xor_sync(0xffffffffu, hi8 ? k4[1] : k4[3], 8));
      const bool hi4 = (lane & 4) != 0;
      double keep = comb(hi4 ? k1 : k0, __shfl_xor_sync(0xffffffffu, hi4 ? k0 : k1, 4));
#pragma unroll
      for (int o = 2; o > 0; o >>= 1) keep = comb(keep, __shfl_xor_sync(0xffffffffu, keep, o));
      return keep;
    }
  }
  if constexpr (K == 1) {
    return warp_sum(v[0]);
  } else if constexpr (K == 2) {
    const bool hi = (lane & 16) != 0;
    double keep = hi ? v[1] : v[0];
    keep += __shfl_xor_sync(0xffffffffu, hi ? v[0] : v[1], 16);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
    return keep;
  } else if constexpr (K == 8) {
    const bool hi = (lane & 16) != 0;
    double k4[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      k4[i] = hi ? v[4 + i] : v[i];
      k4[i] += __shfl_xor_sync(0xffffffffu, hi ? v[i] : v[4 + i], 16);
    }
    const bool hi8 = (lane & 8) != 0;
    double k0 = hi8 ? k4[2] : k4[0], k1 = hi8 ? k4[3] : k4[1];
    k0 += __shfl_xor_sync(0xffffffffu, hi8 ? k4[0] : k4[2], 8);
    k1 += __shfl_xor_sync(0xffffffffu, hi8 ? k4[1] : k4[3], 8);
    const bool hi4 = (lane & 4) != 0;
    double keep = hi4 ? k1 : k0;
    keep += __shfl_xor_sync(0xffffffffu, hi4 ? k0 : k1, 4);
#pragma unroll
    for (int o = 2; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
    return keep;
  } else {
    const bool hi = (lane & 16) != 0;
    double k0 = hi ? v[2] : v[0], k1 = hi ? v[3] : v[1];
    k0 += __shfl_xor_sync(0xffffffffu, hi ? v[0] : v[2], 16);
    k1 += __shfl_xor_sync(0xffffffffu, hi ? v[1] : v[3], 16);
    const bool hi8 = (lane & 8) != 0;
    double keep = hi8 ? k1 : k0;
    keep += __shfl_xor_sync(0xffffffffu, hi8 ? k0 : k1, 8);
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
    return keep;
  }
}

// Ranking state of one warp during a hierarchical sweep: per-lane best, plus the per-lane partial energy
// of an odd top waiting for a partner so that two tops share one reduction.
struct WarpRank {
  Best best;
  double pend;
  int pend_p;  // warp-uniform; 0 = nothing pending
};

// all lanes end up with the warp's best candidate (total order: `better`)
__device__ __forceinline__ Best warp_best(int metric, Best b) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Best other;
    other.key = __shfl_xor_sync(0xffffffffu, b.key, o);
    other.p = __shfl_xor_sync(0xffffffffu, b.p, o);
    if (other.p != 0 && better(metric, other.key, other.p, b)) b = other;
  }
  return b;
}

// 1 / m: table for the small row counts every large period has, a real division otherwise
// (the division is kept out of line: it is almost never taken, and an inlined DDIV sequence at every ranking site
// costs more in code layout than the call)
static __device__ __noinline__ double rcp_slow(int m) { return 1.0 / (double)m; }
__device__ __forceinline__ double rcp_of(const double* rcp, int m) {
  return m < kRcpTab ? rcp[m] : rcp_slow(m);
}

// energy of one candidate from its partial sums: T = sum of S_r^2, A = the part on residues that hold one more sample.
//   full fold:      sum_r S_r^2 / cnt_r          = T / M + (1 / (M + 1) - 1 / M) A      (cnt_r = M, or M + 1 under A)
//   truncated fold: sum_r cnt_r (S_r / M)^2      = T / M + A / M^2                      (S_r over the first M rows only)
template <bool TRUNC>
__device__ __forceinline__ double hier_energy(const double* rcp, int M, double T, double A) {
  const double w = rcp_of(rcp, M);
  if constexpr (TRUNC) return fma(A, w, T) * w;
  else return fma(rcp_of(rcp, M + 1) - w, A, w * T);
}


// Register tiles are deliberately small and come in exactly two shapes -- kTileCols columns for the
// body of a residue range, one column for what is left -- so the hot loops are a few hundred bytes
// of code that every warp of the SM shares.  (A dispatch over 12 tile widths, tried first, lost
// 30 % to instruction-fetch stalls; predicated partial tiles made the compiler spill.)
#ifndef PP_TILECOLS
#define PP_TILECOLS 4
#endif
constexpr int kTileCols = PP_TILECOLS;

// sum of squares of J values as a short tree (no J-long dependent FMA chain)
template <int J>
__device__ __forceinline__ double sum_sq(const double (&v)[J]) {
  if constexpr (J == 1) {
    return v[0] * v[0];
  } else if constexpr (J == 2) {
    return fma(v[1], v[1], v[0] * v[0]);
  } else {
    double lo = v[0] * v[0], hi = v[1] * v[1];
#pragma unroll
    for (int j = 2; j < J; j += 2) {
      lo = fma(v[j], v[j], lo);
      if (j + 1 < J) hi = fma(v[j + 1], v[j + 1], hi);
    }
    return lo + hi;
  }
}

// acc[j] += row[32 j]: the loads of a row are issued together, then the adds
template <int J>
__device__ __forceinline__ void add_row(double (&acc)[J], const double* __restrict__ row) {
  double t[J];
#pragma unroll
  for (int j = 0; j < J; ++j) t[j] = row[32 * j];
#pragma unroll
  for (int j = 0; j < J; ++j) acc[j] += t[j];
}

// acc[j] = sum over `rows` rows (stride p) of row[32 j], added in row order; rows >= 1
template <int J>
__device__ __forceinline__ void fold_rows(double (&acc)[J], const double* __restrict__ ptr, int p, int rows) {
#pragma unroll
  for (int j = 0; j < J; ++j) acc[j] = ptr[32 * j];
#pragma unroll 4
  for (int k = 1; k < rows; ++k) {
    ptr += p;
    add_row<J>(acc, ptr);
  }
}

// ------------------------------------------------------------------------------------------
// direct fold
// ------------------------------------------------------------------------------------------
// One register tile of period p: residues [ra, ra + nres), nres <= 32 J, `rows` rows.
//   Energy / EnergyTail: T += sum S^2;  EnergyTail also C += sum S_r * x[tail_off + r]
//   MaxAbs: T = max(T, |S_r|)
//   Store:  gsS[r] = full-N sum, gsV[r] = S_r * inv   (orthogonalised sweeps)
template <int J, bool PARTIAL, int MODE>
__device__ __forceinline__ void tile_pass(const double* __restrict__ xs, int p, int ra, int nres, int rows,
                                          int tail_off, bool add_tail, double inv, double& T, double& C,
                                          double* __restrict__ gsS, double* __restrict__ gsV) {
  const int lane = threadIdx.x & 31;
  double acc[J];
  fold_rows<J>(acc, xs + ra + lane, p, rows);
  if (MODE == kPassEnergy || MODE == kPassEnergyTail) {
    // lanes past the tile end hold sums of other residues (only possible in a partial tile)
    if (PARTIAL) {
#pragma unroll
      for (int j = 0; j < J; ++j)
        if (lane + 32 * j >= nres) acc[j] = 0.0;
    }
    T += sum_sq<J>(acc);
    if (MODE == kPassEnergyTail) {
#pragma unroll
      for (int j = 0; j < J; ++j) C = fma(acc[j], xs[tail_off + ra + lane + 32 * j], C);
    }
  } else if (MODE == kPassMaxAbs) {
#pragma unroll
    for (int j = 0; j < J; ++j)
      if (lane + 32 * j < nres) T = fmax(T, fabs(acc[j]));
  } else {
#pragma unroll
    for (int j = 0; j < J; ++j) {
      if (lane + 32 * j < nres) {
        const int r = ra + lane + 32 * j;
        gsS[r] = add_tail ? acc[j] + xs[tail_off + r] : acc[j];
        gsV[r] = acc[j] * inv;
      }
    }
  }
}

// residues [lo, hi) of period p: tiles of kTileCols columns, then single columns (the last one masked)
template <int MODE>
__device__ __forceinline__ void fold_range(const double* xs, int p, int lo, int hi, int rows, int tail_off,
                                           bool add_tail, double inv, double& T, double& C, double* gsS,
                                           double* gsV) {
  int ra = lo;
  for (; ra + 32 * kTileCols <= hi; ra += 32 * kTileCols)
    tile_pass<kTileCols, false, MODE>(xs, p, ra, 32 * kTileCols, rows, tail_off, add_tail, inv, T, C, gsS, gsV);
  for (; ra + 64 <= hi; ra += 64)
    tile_pass<2, false, MODE>(xs, p, ra, 64, rows, tail_off, add_tail, inv, T, C, gsS, gsV);
  for (; ra < hi; ra += 32)
    tile_pass<1, true, MODE>(xs, p, ra, min(hi - ra, 32), rows, tail_off, add_tail, inv, T, C, gsS, gsV);
}

// Ranking key of one period, computed by one warp; identical in all lanes.
template <int MODE>
__device__ __forceinline__ double warp_period_key(const SweepParams* sp, int p) {
  const int lane = threadIdx.x & 31;
  const int N = sp->N;
  const bool trunc = sp->trunc != 0;
  const double* xs = staged_window();
  const int M = N / p, rr = N - M * p;
  const int tail_off = M * p;
  const double m = (double)M;
  double TA = 0.0, TB = 0.0, C = 0.0;
  double* gsS = nullptr;
  double* gsV = nullptr;
  if (MODE == kPassStore) {
    gsS = sp->warp_scr + (size_t)(threadIdx.x >> 5) * 2 * sp->pv;
    gsV = gsS + sp->pv;
  }
  // tile A: residues with a sample in the last, partial row
  if (rr > 0) {
    if (MODE == kPassMaxAbs) {
      fold_range<MODE>(xs, p, 0, rr, M + 1, tail_off, false, 0.0, TA, C, gsS, gsV);
    } else {
      fold_range<MODE>(xs, p, 0, rr, trunc ? M : M + 1, tail_off, trunc, trunc ? 1.0 / m : 1.0 / (double)(M + 1), TA,
                       C, gsS, gsV);
    }
  }
  // tile B never has tail samples (and must not read past the short zero pad)
  fold_range<(MODE == kPassEnergyTail ? kPassEnergy : MODE)>(xs, p, rr, p, M, tail_off, false, 1.0 / m,
                                                             (MODE == kPassMaxAbs ? TA : TB), C, gsS, gsV);
  if (MODE == kPassMaxAbs) return warp_max(TA);

  double energy, dot;
  if (MODE == kPassStore) {
    __syncwarp();
    warp_orth_chain_approx(gsV, p, N, trunc, sp->chain_q + sp->chain_off[p], sp->chain_off[p + 1] - sp->chain_off[p]);
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
    // mean = S / M on every residue, counts over all N:  sum cnt * mean^2 = (M (TA + TB) + TA) / M^2
    const double T = TA + TB;
    energy = warp_sum(fma(m, T, TA) / (m * m));
    dot = (MODE == kPassEnergyTail) ? warp_sum((T + C) / m) : energy;
  } else {
    const double w_lo = 1.0 / m, w_diff = 1.0 / (double)(M + 1) - w_lo;
    energy = warp_sum(fma(w_diff, TA, w_lo * (TA + TB)));
    dot = energy;
  }
  if (sp->metric == PP_METRIC_IMPOSED) {
    const double e_res = sp->e_res, sqrtN = sp->sqrtN;
    const double e_trial = fmax(e_res - 2.0 * dot + energy, 0.0);
    return (sqrt(e_res) / sqrtN - sqrt(e_trial) / sqrtN) / sp->data_norm;  // Periods.py:278-280
  }
  return energy;
}

__device__ __forceinline__ double warp_period_key_any(const SweepParams* sp, int p) {
  if (sp->metric == PP_METRIC_MAXABS) return warp_period_key<kPassMaxAbs>(sp, p);
  if (sp->orth) return warp_period_key<kPassStore>(sp, p);
  if (sp->metric == PP_METRIC_IMPOSED && sp->trunc) return warp_period_key<kPassEnergyTail>(sp, p);
  return warp_period_key<kPassEnergy>(sp, p);
}

// ------------------------------------------------------------------------------------------
// hierarchical fold
// ------------------------------------------------------------------------------------------
__host__ __device__ inline int hier_scratch_len(int pmax) { return ((((pmax >> 3) + 2) * 3) / 2 + 3) & ~1; }

// Rows are assigned to the 2^L accumulator sets by (row - M0) mod 2^L, M0 = floor(N / g): the partial
// tail row (row M0, base residues < rr = N mod g) always lands in set 0, the complete rows fill the
// sets cyclically, and at level l (period g 2^l, 2^l sets) the sets with index >= 2^l - (M0 mod 2^l)
// hold one more term on every residue.  A tile therefore covers the whole residue range [0, g) with
// one code path: no split at rr, the tail row is a predicated load.
//
// Riders.  A job with base g and S accumulator sets yields the fold of every period g d, d | S.  With
// S = 3 * 2^LH one pass over the window serves TWO tops: the host q = g 2^LH (g odd, LH in {1, 2}) with its
// chain q/2 .. g, and the rider R = 3 q / 2 or 3 q / 4 (whichever lies in (pmax/2, pmax]) with its chain
// down to 3 g.  About a fifth of the tops ride (the multiples of 3 whose host exists), i.e. a fifth fewer
// passes over the window; the price is a longer level computation per tile.

// energy terms of one level held in `sets` accumulator sets v[0 .. sets): T += sum of squares, A += the part
// whose residues hold one more term (warp-uniform top sets, and set 0 under the tail row)
// MAXABS: T = max |sum| instead (best-correlation metric; counts play no role and A is unused).
// TRUNC (trunc_to_integer_multiple): the candidate only uses its first M = floor(N / p) rows.  The accumulator sets
// hold every complete base row, i.e. `extra` base rows too many for this level: they are the LAST row of each of the
// top `extra` sets (row M0 - SETS + s of set s), so those sets are corrected by one reloaded row (xrow[s * g + 32 j],
// xrow = staged window + (M0 - SETS) g + first residue of the lane) before they are squared; the tail row was never
// accumulated.  The same top sets and tail residues are the ones that hold one more SAMPLE (A) -- there the count,
// not the sum, is what differs.  live[j]: the lane's residue exists (masked tiles run past g).
template <int SETS, int DIM0, int J, bool MAXABS, bool TRUNC = false>
__device__ __forceinline__ void level_energy(const double (&v)[DIM0][J], int extra, const bool (&tail)[J], double& T,
                                             double& A, const double* xrow = nullptr, int g = 0,
                                             const bool* live = nullptr) {
  if constexpr (MAXABS) {
#pragma unroll
    for (int s = 0; s < SETS; ++s)
#pragma unroll
      for (int j = 0; j < J; ++j) T = fmax(T, fabs(v[s][j]));
  } else {
#pragma unroll
    for (int s = 0; s < SETS; ++s) {
      if (s >= SETS - extra) {  // warp-uniform
        double q;
        if constexpr (TRUNC) {
          double t[J];
#pragma unroll
          for (int j = 0; j < J; ++j) t[j] = live[j] ? v[s][j] - xrow[s * g + 32 * j] : 0.0;
          q = sum_sq<J>(t);
        } else {
          q = sum_sq<J>(v[s]);
        }
        T += q;
        A += q;
      } else {
        T += sum_sq<J>(v[s]);
      }
    }
#pragma unroll
    for (int j = 0; j < J; ++j)
      if (tail[j]) A = fma(v[0][j], v[0][j], A);
  }
}

// v[s] += v[s + SETS/2]: the sets of the level with half as many sets
template <int SETS, int DIM0, int J>
__device__ __forceinline__ void level_halve(double (&v)[DIM0][J]) {
#pragma unroll
  for (int s = 0; s < SETS / 2; ++s)
#pragma unroll
    for (int j = 0; j < J; ++j) v[s][j] += v[s + SETS / 2][j];
}

// levels 2^LV .. 1 of a power-of-two set array (compile-time recursion keeps every index static)
// xt (TRUNC only): staged window + first residue of the lane (row 0)
template <int DIM0, int J, int LV, int NL, bool MAXABS, bool TRUNC = false>
struct pow2_levels {
  static __device__ __forceinline__ void run(double (&v)[DIM0][J], int M0, const bool (&tail)[J], double (&T)[NL],
                                             double (&A)[NL], const double* xt = nullptr, int g = 0,
                                             const bool* live = nullptr) {
    constexpr int sets = 1 << LV;
    if constexpr (TRUNC)
      level_energy<sets, DIM0, J, MAXABS, true>(v, M0 & (sets - 1), tail, T[LV], A[LV], xt + (M0 - sets) * g, g, live);
    else
      level_energy<sets, DIM0, J, MAXABS>(v, M0 & (sets - 1), tail, T[LV], A[LV]);
    if constexpr (LV > 0) {
      level_halve<sets, DIM0, J>(v);
      pow2_levels<DIM0, J, LV - 1, NL, MAXABS, TRUNC>::run(v, M0, tail, T, A, xt, g, live);
    }
  }
};
// levels 3 * 2^LV .. 3 of a rider chain
template <int DIM0, int J, int LV, int NL, bool MAXABS, bool TRUNC = false>
struct rider_levels {
  static __device__ __forceinline__ void run(double (&v)[DIM0][J], int M0, const bool (&tail)[J], double (&T)[NL],
                                             double (&A)[NL], const double* xt = nullptr, int g = 0,
                                             const bool* live = nullptr) {
    constexpr int sets = 3 << LV;
    if constexpr (TRUNC)
      level_energy<sets, DIM0, J, MAXABS, true>(v, M0 % sets, tail, T[LV], A[LV], xt + (M0 - sets) * g, g, live);
    else
      level_energy<sets, DIM0, J, MAXABS>(v, M0 % sets, tail, T[LV], A[LV]);
    if constexpr (LV > 0) {
      level_halve<sets, DIM0, J>(v);
      rider_levels<DIM0, J, LV - 1, NL, MAXABS, TRUNC>::run(v, M0, tail, T, A, xt, g, live);
    }
  }
};

// Rows (stride g) of base residues ra + lane + 32 j accumulated into S sets by (row - M0) mod S, plus the
// predicated tail row into set 0.  head = M0 mod S, groups = M0 / S (warp-uniform, computed once per job).
// MASK: the tile may run past g (lanes beyond it are zeroed).
template <int S, int J, bool MASK, bool TRUNC = false>
__device__ __forceinline__ void hier_accumulate(const double* __restrict__ xs, int g, int ra, int M0, int rr, int head,
                                                int groups, double (&acc)[S][J], bool (&tail)[J]) {
  const int lane = threadIdx.x & 31;
  const double* ptr = xs + ra + lane;
  if constexpr (S == 1) {
#pragma unroll
    for (int j = 0; j < J; ++j) acc[0][j] = ptr[32 * j];
    ptr += g;
#pragma unroll 2
    for (int k = 1; k < M0; ++k) {
      add_row<J>(acc[0], ptr);
      ptr += g;
    }
  } else {
    // the first complete group of S rows (rows head .. head + S - 1) initialises the sets, the other groups add,
    // the `head` rows before the first group (sets S - head .. S - 1) come last: no zero fill, no add to zero
    // (every job has at least one complete group: plain tops have N / g >= 2^L, riders are only formed when
    // N / g >= 3 * 2^L, see hier_rider_of)
    const double* hptr = ptr;
    ptr += head * g;
#pragma unroll
    for (int s = 0; s < S; ++s) {
#pragma unroll
      for (int j = 0; j < J; ++j) acc[s][j] = ptr[32 * j];
      ptr += g;
    }
#pragma unroll 1
    for (int i = groups - 1; i > 0; --i) {
#pragma unroll
      for (int s = 0; s < S; ++s) {
        add_row<J>(acc[s], ptr);
        ptr += g;
      }
    }
#pragma unroll
    for (int s = 1; s < S; ++s) {
      if (s >= S - head) {
        add_row<J>(acc[s], hptr);
        hptr += g;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < J; ++j) tail[j] = ra + lane + 32 * j < rr;
  if (!TRUNC && ra < rr) {  // warp-uniform: most tiles of a top lie entirely past the tail row
#pragma unroll
    for (int j = 0; j < J; ++j) {
      double t = 0.0;
      if (tail[j]) t = ptr[32 * j];
      acc[0][j] += t;
    }
  }
  if (MASK) {
#pragma unroll
    for (int j = 0; j < J; ++j) {
      if (ra + lane + 32 * j >= g) {
#pragma unroll
        for (int s = 0; s < S; ++s) acc[s][j] = 0.0;
      }
    }
  }
}

// One register tile of a plain top q = g * 2^L.
template <int L, int J, bool MASK, bool MAXABS, bool TRUNC = false>
__device__ __forceinline__ void hier_tile(const double* __restrict__ xs, int g, int ra, int M0, int rr,
                                          double (&T)[L + 1], double (&A)[L + 1], double* scr) {
  constexpr int S = 1 << L;
  const int lane = threadIdx.x & 31;
  double acc[S][J];
  bool tail[J];
  hier_accumulate<S, J, MASK, TRUNC>(xs, g, ra, M0, rr, M0 & (S - 1), M0 >> L, acc, tail);
  if constexpr (TRUNC) {
    bool live[J];
#pragma unroll
    for (int j = 0; j < J; ++j) live[j] = !MASK || ra + lane + 32 * j < g;
    pow2_levels<S, J, L, L + 1, MAXABS, true>::run(acc, M0, tail, T, A, xs + ra + lane, g, live);
  } else {
    pow2_levels<S, J, L, L + 1, MAXABS>::run(acc, M0, tail, T, A);
  }
  if (scr != nullptr) {
#pragma unroll
    for (int j = 0; j < J; ++j)
      if (!MASK || ra + lane + 32 * j < g) scr[ra + lane + 32 * j] = acc[0][j];
  }
}

// One register tile of a host + rider job: S = 3 * 2^LH sets.  Th/Ah: host levels 2^LH .. 1, Tr/Ar: rider
// levels 3 * 2^(LH-1) .. 3.
template <int LH, int J, bool MASK, bool MAXABS, bool TRUNC = false>
__device__ __forceinline__ void rider_tile(const double* __restrict__ xs, int g, int ra, int M0, int rr, int head,
                                           int groups, double (&Th)[LH + 1], double (&Ah)[LH + 1], double (&Tr)[LH],
                                           double (&Ar)[LH]) {
  constexpr int S = 3 << LH, SH = 1 << LH;
  const int lane = threadIdx.x & 31;
  double acc[S][J];
  bool tail[J];
  hier_accumulate<S, J, MASK, TRUNC>(xs, g, ra, M0, rr, head, groups, acc, tail);
  bool live[J];
#pragma unroll
  for (int j = 0; j < J; ++j) live[j] = !MASK || ra + lane + 32 * j < g;
  const double* xt = xs + ra + lane;
  {  // host chain: sets t, t + SH, t + 2 SH fold into level SH (set t = rows with (row - M0) mod SH == t)
    double hv[SH][J];
#pragma unroll
    for (int t = 0; t < SH; ++t)
#pragma unroll
      for (int j = 0; j < J; ++j) hv[t][j] = (acc[t][j] + acc[t + SH][j]) + acc[t + 2 * SH][j];
    if constexpr (TRUNC) pow2_levels<SH, J, LH, LH + 1, MAXABS, true>::run(hv, M0, tail, Th, Ah, xt, g, live);
    else pow2_levels<SH, J, LH, LH + 1, MAXABS>::run(hv, M0, tail, Th, Ah);
  }
  level_halve<S, S, J>(acc);  // level 3 * 2^(LH-1)
  if constexpr (TRUNC) rider_levels<S, J, LH - 1, LH, MAXABS, true>::run(acc, M0, tail, Tr, Ar, xt, g, live);
  else rider_levels<S, J, LH - 1, LH, MAXABS>::run(acc, M0, tail, Tr, Ar);
}

// register columns per accumulator set of a hierarchical tile: 8 accumulators per lane (8 / 4 / 2 / 1 columns
// for L = 0..3).  16 accumulators halve the number of tiles of L >= 1 but measured 1.4 % slower: the larger
// tile bodies cost more in instruction fetch than the saved per-tile overhead (ncu: 9 % of the stall samples
// are no_instruction once the rider tiles are in the kernel).
#ifndef PP_HIER_ACCS
#define PP_HIER_ACCS 8
#endif
template <int L>
struct hier_cols {
  static constexpr int value = (PP_HIER_ACCS >> L) < 8 ? (PP_HIER_ACCS >> L) : 8;
};

// One top period q = g * 2^L and every candidate q / 2^k below it.  Non-trunc, non-orth, NORM / GAMMA.
template <int L, bool MAXABS, bool TRUNC = false>
__device__ __forceinline__ void warp_hier_top_L(RankCtx rc, int g, int M0, int rr, double* scr, WarpRank& wr) {
  // M0 = floor(N / g) complete base rows; base residues below rr = N - M0 g have one more (tail) row
  constexpr int J = hier_cols<L>::value;
  const int lane = threadIdx.x & 31;
  const int N = rc.N;
  const double* xs = staged_window();
  const bool chain = (L == 3) && !(g & 1) && (g >> 1) >= rc.pmin;
  double* out = chain ? scr : nullptr;
  double T[L + 1], A[L + 1];
#pragma unroll
  for (int i = 0; i <= L; ++i) T[i] = A[i] = 0.0;
  int ra = 0;
  for (; ra + 32 * J <= g; ra += 32 * J) hier_tile<L, J, false, MAXABS, TRUNC>(xs, g, ra, M0, rr, T, A, out);
  if constexpr (J > 2)
    for (; ra + 64 <= g; ra += 64) hier_tile<L, 2, false, MAXABS, TRUNC>(xs, g, ra, M0, rr, T, A, out);
  for (; ra < g; ra += 32) hier_tile<L, 1, true, MAXABS, TRUNC>(xs, g, ra, M0, rr, T, A, out);
  // per-lane partial energies of the L + 1 levels, reduced together
  constexpr int KP = L == 0 ? 1 : (L == 1 ? 2 : 4);
  double e[KP];
#pragma unroll
  for (int i = 0; i < KP; ++i) {
    if (i <= L) {
      if constexpr (MAXABS) {
        e[i] = T[i];
      } else {
        e[i] = hier_energy<TRUNC>(rc.rcp, M0 >> i, T[i], A[i]);
      }
    } else {
      e[i] = 0.0;
    }
  }
  if constexpr (L == 0) {
    if (wr.pend_p == 0) {  // wait for the next odd top
      wr.pend = e[0];
      wr.pend_p = g;
    } else {
      const double pair[2] = {wr.pend, e[0]};
      const double key = warp_sum_multi<2, MAXABS>(pair);
      consider_lane(rc, key, (lane & 16) ? g : wr.pend_p, (lane & 15) == 0, wr.best);
      wr.pend_p = 0;
    }
  } else {
    const double key = warp_sum_multi<KP, MAXABS>(e);
    constexpr int shift = KP == 2 ? 4 : 3;
    const int k = lane >> shift;
    consider_lane(rc, key, k <= L ? (g << k) : 0, (lane & ((1 << shift) - 1)) == 0, wr.best);
  }
  Best& best = wr.best;
  if (chain) {
    __syncwarp();
    double* src = scr;
    double* dst = scr + ((g + 1) & ~1);
    int h = g;
    while (!(h & 1) && (h >> 1) >= rc.pmin) {
      const int h2 = h >> 1;
      const int M = N / h2, r0h = N - M * h2;
      // truncated fold: the halves hold 2 floor(M / 2) rows of period h2; an odd M brings one more complete row
      const double* odd_row = (TRUNC && (M & 1)) ? xs + (M - 1) * h2 : nullptr;
      double t = 0.0, a = 0.0;
      for (int r = lane; r < h2; r += 32) {
        double v = src[r] + src[r + h2];
        if (TRUNC && odd_row != nullptr) v += odd_row[r];
        dst[r] = v;
        if constexpr (MAXABS) {
          t = fmax(t, fabs(v));
        } else {
          t = fma(v, v, t);
          if (r < r0h) a = fma(v, v, a);
        }
      }
      __syncwarp();
      if constexpr (MAXABS) consider(rc, warp_max(t), h2, best);
      else consider(rc, warp_sum(hier_energy<TRUNC>(rc.rcp, M, t, a)), h2, best);
      double* swp = src;
      src = dst;
      dst = swp;
      h = h2;
    }
    __syncwarp();
  }
}

// A host top q = g 2^LH (g odd) together with its rider; candidates g 2^i (i <= LH) and 3 g 2^i (i < LH) that
// lie in [pmin, pmax].
template <int LH, bool MAXABS, bool TRUNC = false>
__device__ __forceinline__ void warp_hier_rider_L(RankCtx rc, int g, int M0, int rr, WarpRank& wr) {
  constexpr int S = 3 << LH;
#ifndef PP_RIDER_J1
#define PP_RIDER_J1 2
#endif
  constexpr int J = LH == 1 ? PP_RIDER_J1 : 2;
  const int lane = threadIdx.x & 31;
  const double* xs = staged_window();
  const int head = M0 % S, groups = M0 / S;
  double Th[LH + 1], Ah[LH + 1], Tr[LH], Ar[LH];
#pragma unroll
  for (int i = 0; i <= LH; ++i) Th[i] = Ah[i] = 0.0;
#pragma unroll
  for (int i = 0; i < LH; ++i) Tr[i] = Ar[i] = 0.0;
  int ra = 0;
  for (; ra + 32 * J <= g; ra += 32 * J)
    rider_tile<LH, J, false, MAXABS, TRUNC>(xs, g, ra, M0, rr, head, groups, Th, Ah, Tr, Ar);
  if constexpr (J > 2)
    for (; ra + 64 <= g; ra += 64) rider_tile<LH, 2, false, MAXABS, TRUNC>(xs, g, ra, M0, rr, head, groups, Th, Ah, Tr, Ar);
  for (; ra < g; ra += 32) rider_tile<LH, 1, true, MAXABS, TRUNC>(xs, g, ra, M0, rr, head, groups, Th, Ah, Tr, Ar);
  // values 0 .. LH: host levels g 2^i; values LH+1 .. 2 LH: rider levels 3 g 2^i
  constexpr int NV = 2 * LH + 1;          // 3 or 5
  constexpr int KP = NV <= 4 ? 4 : 8;
  double e[KP];
#pragma unroll
  for (int i = 0; i < KP; ++i) e[i] = 0.0;
#pragma unroll
  for (int i = 0; i <= LH; ++i) {
    if constexpr (MAXABS) {
      e[i] = Th[i];
    } else {
      e[i] = hier_energy<TRUNC>(rc.rcp, M0 >> i, Th[i], Ah[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < LH; ++i) {
    if constexpr (MAXABS) {
      e[LH + 1 + i] = Tr[i];
    } else {
      e[LH + 1 + i] = hier_energy<TRUNC>(rc.rcp, M0 / (3 << i), Tr[i], Ar[i]);
    }
  }
  const double key = warp_sum_multi<KP, MAXABS>(e);
  constexpr int shift = KP == 4 ? 3 : 2;
  const int k = lane >> shift;
  int p = 0;
  if (k <= LH) p = g << k;
  else if (k < NV) p = (3 * g) << (k - LH - 1);
  if (p < rc.pmin || p > rc.pmax) p = 0;
  consider_lane(rc, key, p, (lane & ((1 << shift) - 1)) == 0, wr.best);
}

// ------------------------------------------------------------------------------------------
// fp32 nomination sweep
// ------------------------------------------------------------------------------------------
// The same jobs (tops, chains, riders) evaluated in float: a lane owns the residue PAIR ra + 2 lane + 64 j + {0, 1},
// one aligned LDS.64 feeds one FADD2, so a pass costs half the shared-memory wavefronts and half the
// instructions of the fp64 pass.  The float energies only NOMINATE: cta_sweep re-evaluates every candidate whose
// upper bound reaches the best lower bound with the sequential fp64 fold, so the selected period and its norm are
// those of the exact fold (pp_sweep.cuh: cta_sweep).
struct F32Window {
  int off0;  // byte offset in pp_smem of x0[n] = (float) x[n]
  int off1;  // byte offset in pp_smem of x1[n] = (float) x[n + 1]
  // byte offset of the aligned pair (e + 2 lane, e + 2 lane + 1), e = element index of the pair owned by lane 0
  __device__ __forceinline__ int pair_byte(int e) const {
    return ((e & 1) ? off1 + 4 * (e - 1) : off0 + 4 * e) + 8 * (threadIdx.x & 31);
  }
};

// Blackwell's packed single-precision add (add.rn.f32x2, SASS FADD2): one instruction for the residue pair a lane
// owns -- the row loop of the float sweep is one LDS.64 and one FADD2 per 64 residues of a warp
__device__ __forceinline__ float2 add_f32x2(float2 a, float2 b) {
#ifndef PP_NO_F32X2
  unsigned long long ra, rb, rd;
  ra = *reinterpret_cast<unsigned long long*>(&a);
  rb = *reinterpret_cast<unsigned long long*>(&b);
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  return *reinterpret_cast<float2*>(&rd);
#else
  return make_float2(a.x + b.x, a.y + b.y);
#endif
}

template <int J>
__device__ __forceinline__ void add_row_f32(float2 (&acc)[J], const float2* __restrict__ row) {
  float2 t[J];
#pragma unroll
  for (int j = 0; j < J; ++j) t[j] = row[32 * j];
#pragma unroll
  for (int j = 0; j < J; ++j) acc[j] = add_f32x2(acc[j], t[j]);
}

__device__ __forceinline__ float2 fma_f32x2(float2 a, float2 b, float2 c) {
#ifndef PP_NO_F32X2
  unsigned long long ra, rb, rc, rd;
  ra = *reinterpret_cast<unsigned long long*>(&a);
  rb = *reinterpret_cast<unsigned long long*>(&b);
  rc = *reinterpret_cast<unsigned long long*>(&c);
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  return *reinterpret_cast<float2*>(&rd);
#else
  return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y));
#endif
}

template <int J>
__device__ __forceinline__ float sum_sq_f32(const float2 (&v)[J]) {
  float2 acc = make_float2(v[0].x * v[0].x, v[0].y * v[0].y);
#pragma unroll
  for (int j = 1; j < J; ++j) acc = fma_f32x2(v[j], v[j], acc);   // same two chains as the scalar form
  return acc.x + acc.y;
}

template <int SETS, int DIM0, int J>
__device__ __forceinline__ void level_energy_f32(const float2 (&v)[DIM0][J], int extra, const bool (&tail)[J][2], float& T,
                                                 float& A) {
#pragma unroll
  for (int s = 0; s < SETS; ++s) {
    const float q = sum_sq_f32<J>(v[s]);
    T += q;
    if (s >= SETS - extra) A += q;  // warp-uniform
  }
#pragma unroll
  for (int j = 0; j < J; ++j) {
    if (tail[j][0]) A = fmaf(v[0][j].x, v[0][j].x, A);
    if (tail[j][1]) A = fmaf(v[0][j].y, v[0][j].y, A);
  }
}
template <int SETS, int DIM0, int J>
__device__ __forceinline__ void level_halve_f32(float2 (&v)[DIM0][J]) {
#pragma unroll
  for (int s = 0; s < SETS / 2; ++s)
#pragma unroll
    for (int j = 0; j < J; ++j) v[s][j] = add_f32x2(v[s][j], v[s + SETS / 2][j]);
}
template <int DIM0, int J, int LV, int NL>
struct pow2_levels_f32 {
  static __device__ __forceinline__ void run(float2 (&v)[DIM0][J], int M0, const bool (&tail)[J][2], float (&T)[NL],
                                             float (&A)[NL]) {
    constexpr int sets = 1 << LV;
    level_energy_f32<sets, DIM0, J>(v, M0 & (sets - 1), tail, T[LV], A[LV]);
    if constexpr (LV > 0) {
      level_halve_f32<sets, DIM0, J>(v);
      pow2_levels_f32<DIM0, J, LV - 1, NL>::run(v, M0, tail, T, A);
    }
  }
};
template <int DIM0, int J, int LV, int NL>
struct rider_levels_f32 {
  static __device__ __forceinline__ void run(float2 (&v)[DIM0][J], int M0, const bool (&tail)[J][2], float (&T)[NL],
                                             float (&A)[NL]) {
    constexpr int sets = 3 << LV;
    level_energy_f32<sets, DIM0, J>(v, M0 % sets, tail, T[LV], A[LV]);
    if constexpr (LV > 0) {
      level_halve_f32<sets, DIM0, J>(v);
      rider_levels_f32<DIM0, J, LV - 1, NL>::run(v, M0, tail, T, A);
    }
  }
};

// rows (stride g) of the base-residue pairs ra + 2 lane + 64 j + {0, 1} into S sets by (row - M0) mod S, plus the
// tail row into set 0; lanes / components past g are zeroed when MASK.  As in hier_accumulate, the first complete
// group of S rows initialises the sets (no zero fill) and the `head` rows before it come last.
// Row k starts at element ra + k g: its pair sits at (k odd ? po : pe) + 4 k g bytes.  For even g both are the same
// copy of the window; for odd g the rows alternate between the two copies.  So rows of one parity are one pointer
// that advances 8 g bytes per row, and every row costs one LDS.64 per column plus one address add.
template <int J>
__device__ __forceinline__ void load_row_f32(float2 (&acc)[J], const unsigned char* row) {
  const float2* r = reinterpret_cast<const float2*>(row);
#pragma unroll
  for (int j = 0; j < J; ++j) acc[j] = r[32 * j];
}
template <int S, int J, bool MASK>
__device__ __forceinline__ void hier_accumulate_f32(const F32Window& w, int g, int ra, int M0, int rr, int head,
                                                    int groups, float2 (&acc)[S][J], bool (&tail)[J][2]) {
  const int lane = threadIdx.x & 31;
  const int g4 = 4 * g, g8 = 8 * g;
  const unsigned char* pe = pp_smem + w.pair_byte(ra);
  const unsigned char* po = pp_smem + w.pair_byte(ra + g) - g4;
  const unsigned char* tail_row;
  if constexpr (S == 1) {
    load_row_f32<J>(acc[0], pe);
    const unsigned char* qo = po + g4;  // row 1
    const unsigned char* qe = pe + g8;  // row 2
#pragma unroll 1
    for (int k = (M0 - 1) >> 1; k > 0; --k) {
      add_row_f32<J>(acc[0], reinterpret_cast<const float2*>(qo));
      add_row_f32<J>(acc[0], reinterpret_cast<const float2*>(qe));
      qo += g8;
      qe += g8;
    }
    if (!(M0 & 1)) add_row_f32<J>(acc[0], reinterpret_cast<const float2*>(qo));  // row M0 - 1
    tail_row = (M0 & 1) ? qo : qe;
  } else {  // S is even
    const unsigned char* qe = ((head & 1) ? po : pe) + head * g4;  // rows head + even s
    const unsigned char* qo = ((head & 1) ? pe : po) + (head + 1) * g4;  // rows head + odd s
#pragma unroll
    for (int s = 0; s < S; ++s) {
      if (s & 1) {
        load_row_f32<J>(acc[s], qo);
        qo += g8;
      } else {
        load_row_f32<J>(acc[s], qe);
        qe += g8;
      }
    }
#pragma unroll 1
    for (int i = groups - 1; i > 0; --i) {
#pragma unroll
      for (int s = 0; s < S; ++s) {
        if (s & 1) {
          add_row_f32<J>(acc[s], reinterpret_cast<const float2*>(qo));
          qo += g8;
        } else {
          add_row_f32<J>(acc[s], reinterpret_cast<const float2*>(qe));
          qe += g8;
        }
      }
    }
    const unsigned char* hc = pe;       // head rows 0, 1, ... into sets S - head .. S - 1
    const unsigned char* hn = po + g4;
#pragma unroll
    for (int s = 1; s < S; ++s) {
      if (s >= S - head) {  // warp-uniform
        add_row_f32<J>(acc[s], reinterpret_cast<const float2*>(hc));
        const unsigned char* t = hn;
        hn = hc + g8;
        hc = t;
      }
    }
    tail_row = qe;  // row head + groups S = M0
  }
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int r = ra + 2 * lane + 64 * j;
    tail[j][0] = r < rr;
    tail[j][1] = r + 1 < rr;
  }
  if (ra < rr) {  // warp-uniform
    // one predicate per pair: the tail row of a pair starting below rr may reach element N, which is zero in both
    // copies; the pair of a residue >= rr can lie past the zero pad
    const float2* row = reinterpret_cast<const float2*>(tail_row);
#pragma unroll
    for (int j = 0; j < J; ++j) {
      float2 t = make_float2(0.f, 0.f);
      if (tail[j][0]) t = row[32 * j];
      acc[0][j] = add_f32x2(acc[0][j], t);
    }
  }
  if (MASK) {
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int r = ra + 2 * lane + 64 * j;
#pragma unroll
      for (int s = 0; s < S; ++s) {
        if (r >= g) acc[s][j].x = 0.f;
        if (r + 1 >= g) acc[s][j].y = 0.f;
      }
    }
  }
}

// per-tile float partial energies go into double accumulators (the sum over tiles is then exact enough to ignore)
template <int NL>
__device__ __forceinline__ void fold_partial(double (&T)[NL], double (&A)[NL], const float (&t)[NL], const float (&a)[NL]) {
#pragma unroll
  for (int i = 0; i < NL; ++i) {
    T[i] += (double)t[i];
    A[i] += (double)a[i];
  }
}

template <int L, int J, bool MASK>
__device__ __forceinline__ void hier_tile_f32(const F32Window& w, int g, int ra, int M0, int rr, double (&T)[L + 1],
                                              double (&A)[L + 1], double* scr) {
  constexpr int S = 1 << L;
  const int lane = threadIdx.x & 31;
  float2 acc[S][J];
  bool tail[J][2];
  hier_accumulate_f32<S, J, MASK>(w, g, ra, M0, rr, M0 & (S - 1), M0 >> L, acc, tail);
  float t[L + 1], a[L + 1];
#pragma unroll
  for (int i = 0; i <= L; ++i) t[i] = a[i] = 0.f;
  pow2_levels_f32<S, J, L, L + 1>::run(acc, M0, tail, t, a);
  fold_partial<L + 1>(T, A, t, a);
  if (scr != nullptr) {
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int r = ra + 2 * lane + 64 * j;
      if (r < g) scr[r] = (double)acc[0][j].x;
      if (r + 1 < g) scr[r + 1] = (double)acc[0][j].y;
    }
  }
}

template <int LH, int J, bool MASK>
__device__ __forceinline__ void rider_tile_f32(const F32Window& w, int g, int ra, int M0, int rr, int head, int groups,
                                               double (&Th)[LH + 1], double (&Ah)[LH + 1], double (&Tr)[LH],
                                               double (&Ar)[LH]) {
  constexpr int S = 3 << LH, SH = 1 << LH;
  float2 acc[S][J];
  bool tail[J][2];
  hier_accumulate_f32<S, J, MASK>(w, g, ra, M0, rr, head, groups, acc, tail);
  {
    float2 hv[SH][J];
#pragma unroll
    for (int t = 0; t < SH; ++t)
#pragma unroll
      for (int j = 0; j < J; ++j) {
        hv[t][j].x = (acc[t][j].x + acc[t + SH][j].x) + acc[t + 2 * SH][j].x;
        hv[t][j].y = (acc[t][j].y + acc[t + SH][j].y) + acc[t + 2 * SH][j].y;
      }
    float t[LH + 1], a[LH + 1];
#pragma unroll
    for (int i = 0; i <= LH; ++i) t[i] = a[i] = 0.f;
    pow2_levels_f32<SH, J, LH, LH + 1>::run(hv, M0, tail, t, a);
    fold_partial<LH + 1>(Th, Ah, t, a);
  }
  level_halve_f32<S, S, J>(acc);
  float t[LH], a[LH];
#pragma unroll
  for (int i = 0; i < LH; ++i) t[i] = a[i] = 0.f;
  rider_levels_f32<S, J, LH - 1, LH>::run(acc, M0, tail, t, a);
  fold_partial<LH>(Tr, Ar, t, a);
}

// columns (of 64 residues) per accumulator set: 16 float accumulators per lane (8 / 4 / 2 / 1 columns for L = 0..3),
// the register budget of the fp64 tiles, so a float tile covers twice their residues.  What is left of a top after
// the full tiles runs as masked tiles of half the width (one or two of them).
template <int L>
struct hier_cols_f32 {
  static constexpr int value = (8 >> L) > 1 ? (8 >> L) : 1;
};
constexpr int kRiderColsF32 = 2;  // rider tiles: 3 * 2^LH sets of 2 columns

// float energies of one top and its chain, written to keys[] (no ranking here)
template <int L>
__device__ __forceinline__ void warp_hier_top_f32(const RankCtx& rc, const F32Window& w, double* keys, int g, int M0,
                                                  int rr, double* scr, double& pend, int& pend_p) {
  constexpr int J = hier_cols_f32<L>::value;
  const int lane = threadIdx.x & 31;
  const int N = rc.N;
  const bool chain = (L == 3) && !(g & 1) && (g >> 1) >= rc.pmin;
  double* out = chain ? scr : nullptr;
  double T[L + 1], A[L + 1];
#pragma unroll
  for (int i = 0; i <= L; ++i) T[i] = A[i] = 0.0;
  int ra = 0;
  constexpr int JR = J > 1 ? J / 2 : 1;
  for (; ra + 64 * J <= g; ra += 64 * J) hier_tile_f32<L, J, false>(w, g, ra, M0, rr, T, A, out);
  for (; ra < g; ra += 64 * JR) hier_tile_f32<L, JR, true>(w, g, ra, M0, rr, T, A, out);
  constexpr int KP = L == 0 ? 1 : (L == 1 ? 2 : 4);
  double e[KP];
#pragma unroll
  for (int i = 0; i < KP; ++i) {
    if (i <= L) {
      const int M = M0 >> i;
      const double w_lo = rcp_of(rc.rcp, M), w_diff = rcp_of(rc.rcp, M + 1) - w_lo;
      e[i] = fma(w_diff, A[i], w_lo * T[i]);
    } else {
      e[i] = 0.0;
    }
  }
  if constexpr (L == 0) {
    if (pend_p == 0) {
      pend = e[0];
      pend_p = g;
    } else {
      const double pair[2] = {pend, e[0]};
      const double key = warp_sum_multi<2>(pair);
      if ((lane & 15) == 0) keys[(lane & 16) ? g : pend_p] = key;
      pend_p = 0;
    }
  } else {
    const double key = warp_sum_multi<KP>(e);
    constexpr int shift = KP == 2 ? 4 : 3;
    const int k = lane >> shift;
    if ((lane & ((1 << shift) - 1)) == 0 && k <= L) keys[g << k] = key;
  }
  if (chain) {
    __syncwarp();
    double* src = scr;
    double* dst = scr + ((g + 1) & ~1);
    int h = g;
    while (!(h & 1) && (h >> 1) >= rc.pmin) {
      const int h2 = h >> 1;
      const int M = N / h2, r0h = N - M * h2;
      const double w_lo = rcp_of(rc.rcp, M), w_diff = rcp_of(rc.rcp, M + 1) - w_lo;
      double t = 0.0, a = 0.0;
      for (int r = lane; r < h2; r += 32) {
        const double v = src[r] + src[r + h2];
        dst[r] = v;
        t = fma(v, v, t);
        if (r < r0h) a = fma(v, v, a);
      }
      __syncwarp();
      const double key = warp_sum(fma(w_diff, a, w_lo * t));
      if (lane == 0) keys[h2] = key;
      double* swp = src;
      src = dst;
      dst = swp;
      h = h2;
    }
    __syncwarp();
  }
}

template <int LH>
__device__ __forceinline__ void warp_hier_rider_f32(const RankCtx& rc, const F32Window& w, double* keys, int g, int M0,
                                                    int rr) {
  constexpr int S = 3 << LH;
  const int lane = threadIdx.x & 31;
  const int head = M0 % S, groups = M0 / S;
  double Th[LH + 1], Ah[LH + 1], Tr[LH], Ar[LH];
#pragma unroll
  for (int i = 0; i <= LH; ++i) Th[i] = Ah[i] = 0.0;
#pragma unroll
  for (int i = 0; i < LH; ++i) Tr[i] = Ar[i] = 0.0;
  int ra = 0;
  constexpr int J = kRiderColsF32;
  for (; ra + 64 * J <= g; ra += 64 * J) rider_tile_f32<LH, J, false>(w, g, ra, M0, rr, head, groups, Th, Ah, Tr, Ar);
  for (; ra < g; ra += 64) rider_tile_f32<LH, 1, true>(w, g, ra, M0, rr, head, groups, Th, Ah, Tr, Ar);
  constexpr int NV = 2 * LH + 1;
  constexpr int KP = NV <= 4 ? 4 : 8;
  double e[KP];
#pragma unroll
  for (int i = 0; i < KP; ++i) e[i] = 0.0;
#pragma unroll
  for (int i = 0; i <= LH; ++i) {
    const int M = M0 >> i;
    const double w_lo = rcp_of(rc.rcp, M), w_diff = rcp_of(rc.rcp, M + 1) - w_lo;
    e[i] = fma(w_diff, Ah[i], w_lo * Th[i]);
  }
#pragma unroll
  for (int i = 0; i < LH; ++i) {
    const int M = M0 / (3 << i);
    const double w_lo = rcp_of(rc.rcp, M), w_diff = rcp_of(rc.rcp, M + 1) - w_lo;
    e[LH + 1 + i] = fma(w_diff, Ar[i], w_lo * Tr[i]);
  }
  const double key = warp_sum_multi<KP>(e);
  constexpr int shift = KP == 4 ? 3 : 2;
  const int k = lane >> shift;
  int p = 0;
  if (k <= LH) p = g << k;
  else if (k < NV) p = (3 * g) << (k - LH - 1);
  if (p < rc.pmin || p > rc.pmax) p = 0;
  if (p != 0 && (lane & ((1 << shift) - 1)) == 0) keys[p] = key;
}

__device__ __forceinline__ void warp_hier_job_f32(const RankCtx& rc, const F32Window& w, double* keys, uint2 e, double* scr,
                                                  double& pend, int& pend_p) {
  const int g = e.x & 0xffff, L = (e.x >> 16) & 0xf, M0 = e.y & 0xffff, rr = e.y >> 16;
  if (e.x >> 20) {
    if (L == 1) warp_hier_rider_f32<1>(rc, w, keys, g, M0, rr);
    else warp_hier_rider_f32<2>(rc, w, keys, g, M0, rr);
    return;
  }
  switch (L) {
    case 0: warp_hier_top_f32<0>(rc, w, keys, g, M0, rr, scr, pend, pend_p); break;
    case 1: warp_hier_top_f32<1>(rc, w, keys, g, M0, rr, scr, pend, pend_p); break;
    case 2: warp_hier_top_f32<2>(rc, w, keys, g, M0, rr, scr, pend, pend_p); break;
    default: warp_hier_top_f32<3>(rc, w, keys, g, M0, rr, scr, pend, pend_p); break;
  }
}

// Upper bound of |float key - exact energy| of candidate p.  c = ceil(N/p), M = floor(N/p), u = 2^-24, e >= sum x^2 of
// the swept signal, K = kF32TileTerms: the float terms one lane sums per tile and level (2 components x J columns x
// S sets of that level).
//   residue sums  S_r adds its c_r <= c samples in float, in any order, after rounding them to float:
//                 |dS_r| <= c_r u A_r with A_r = sum_{i in r} |x_i|, so |d(S_r^2 / c_r)| <= 2 u A_r^2 <= 2 c u e_r
//                 (Cauchy-Schwarz: A_r^2 <= c_r e_r, e_r = sum_{i in r} x_i^2), 2 c u e over all residues;
//   tile sums     a tile's float T and A of one level each sum at most K rounded squares (relative error K u); the
//                 key T / M + (1/(M+1) - 1/M) A then moves by K u (T / M + A / (M (M+1))) <= K u (M + 2) / M E,
//                 since T <= (M + 1) E and A <= T, with E <= e the candidate's energy;
//   underflow     gradual underflow adds at most 2^-150 to each rounded sample and square (float sums round exactly
//                 below 2^-126): 2^-149 (sum |x| + p) <= 2^-149 (N + e + p).
// The tile partials are summed and weighted in double, which the doubling of this first-order bound covers.  Every
// float value stays below c e <= N e, so the caller must keep N e below the float range (mbest_kernel: 2^120).
constexpr int kF32TileTerms = 24;
static_assert(2 * 8 <= kF32TileTerms && 2 * (1 << 2) * kRiderColsF32 <= kF32TileTerms &&
                  2 * (3 << 1) * kRiderColsF32 <= kF32TileTerms,
              "tops hold 8 pairs per lane and level, riders 2^LH (host) or 3 * 2^(LH-1) (rider) sets of pairs");
__device__ __forceinline__ double f32_energy_tol(int N, int p, double e) {
  const double u = 0x1p-24;
  const int M = N / p, c = (N + p - 1) / p;
  const double terms = 2.0 * (double)c + (double)kF32TileTerms * (double)(M + 2) / (double)M;
  return 2.0 * (terms * u * e + 0x1p-149 * ((double)N + (double)p + e));
}

// ------------------------------------------------------------------------------------------
// job table
// ------------------------------------------------------------------------------------------
// Descriptor of one job: x = g | L << 16 | rider << 20, y = floor(N / g) | (N mod g) << 16.
// Built once per launch in hand-out order: grouped by class (plain L = 0..3, then hosts with a rider) so
// that all warps of an SM run the same specialisation at the same time, ascending q inside a class.
// (Handing out the long rider jobs FIRST measured 12 % slower.)
__host__ __device__ inline int hier_ctz(int v) {
  int c = 0;
  while (!(v & 1) && c < 30) {
    v >>= 1;
    ++c;
  }
  return c;
}
__host__ __device__ inline int hier_top_lo(int pmin, int pmax) {
  return pmin > (pmax >> 1) + 1 ? pmin : (pmax >> 1) + 1;
}
// upper bound on the number of jobs (= number of tops)
__host__ __device__ inline int hier_top_count(int pmin, int pmax) {
  const int top_lo = hier_top_lo(pmin, pmax);
  return pmax >= top_lo ? pmax - top_lo + 1 : 0;
}
__host__ __device__ inline int hier_level(int t, int pmin) {
  int L = hier_ctz(t);
  if (L > 3) L = 3;
  while (L > 0 && (t >> L) < pmin) --L;
  return L;
}
// the top that rides on host q, or 0
__host__ __device__ inline int hier_rider_of(int N, int q, int pmin, int pmax, bool riders) {
  if (!riders) return 0;
  const int L = hier_level(q, pmin);
  if (L < 1 || L > 2 || hier_ctz(q) != L) return 0;  // host classes: q = 2 g or 4 g, g odd
  if (N / (q >> L) < (3 << L)) return 0;             // fewer rows than accumulator sets: no complete group
  int R;
  if (3 * q <= 2 * pmax) R = 3 * q / 2;
  else if (L == 2) R = 3 * q / 4;
  else return 0;
  if (R < hier_top_lo(pmin, pmax) || R > pmax) return 0;
  if (hier_level(R, pmin) != hier_ctz(R)) return 0;  // the rider's own chain is exactly 3 g 2^i
  return R;
}
constexpr int kHierRiderMaxTops = 4096;  // rider matching runs in one CTA with two ints of shared memory per top

// number of jobs the table will hold (host-side mirror of tops_kernel)
inline int hier_job_count(int N, int pmin, int pmax, bool riders) {
  const int n = hier_top_count(pmin, pmax);
  if (!riders || n > kHierRiderMaxTops) return n;
  const int lo = hier_top_lo(pmin, pmax);
  int jobs = n;
  for (int q = lo; q <= pmax; ++q)
    if (hier_rider_of(N, q, pmin, pmax, true)) --jobs;
  return jobs;
}

// one CTA; dynamic shared memory: 2 ints per top
static __global__ void tops_kernel(int N, int pmin, int pmax, int riders, uint2* __restrict__ tops) {
  extern __shared__ int tk_smem[];
  const int lo = hier_top_lo(pmin, pmax);
  const int n = pmax >= lo ? pmax - lo + 1 : 0;
  int* rider = tk_smem;      // rider[t - lo]: the top riding on t (0: none)
  int* cls = tk_smem + n;    // cls[t - lo]: hand-out class of t, -1 if t rides on another top
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    rider[i] = hier_rider_of(N, lo + i, pmin, pmax, riders != 0);
    cls[i] = 0;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    if (rider[i]) cls[rider[i] - lo] = -1;  // each top rides on at most one host
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    if (cls[i] == 0) cls[i] = rider[i] ? 4 + hier_level(lo + i, pmin) : hier_level(lo + i, pmin);
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int c = cls[i];
    if (c < 0) continue;
    int rank = 0;
    for (int u = 0; u < n; ++u) {
      const int cu = cls[u];
      rank += (cu >= 0) && (cu < c || (cu == c && u < i));
    }
    const int q = lo + i, L = hier_level(q, pmin);
    const int g = q >> L, M0 = N / g, rr = N - M0 * g;
    tops[rank] = make_uint2((unsigned)g | ((unsigned)L << 16) | ((rider[i] ? 1u : 0u) << 20),
                            (unsigned)M0 | ((unsigned)rr << 16));
  }
}

// Build the job table in the caller-provided buffer (>= hier_top_count entries) on `stream`; returns the
// number of jobs.
inline int build_hier_jobs(int N, int pmin, int pmax, bool want_riders, uint2* tops, cudaStream_t stream) {
  const int n = hier_top_count(pmin, pmax);
  if (n <= 0) return 0;
  const bool riders = n <= kHierRiderMaxTops && want_riders;
  const size_t smem = (size_t)2 * n * sizeof(int);
  if (smem > 48 * 1024)
    cudaFuncSetAttribute(tops_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  tops_kernel<<<1, 512, smem, stream>>>(N, pmin, pmax, riders ? 1 : 0, tops);
  return hier_job_count(N, pmin, pmax, riders);
}

template <bool MAXABS, bool TRUNC = false>
__device__ __forceinline__ void warp_hier_top(const RankCtx& rc, uint2 e, double* scr, WarpRank& wr) {
  const int g = e.x & 0xffff, L = (e.x >> 16) & 0xf, M0 = e.y & 0xffff, rr = e.y >> 16;
#ifndef PP_NO_RIDERS
  if (e.x >> 20) {
    if (L == 1) warp_hier_rider_L<1, MAXABS, TRUNC>(rc, g, M0, rr, wr);
    else warp_hier_rider_L<2, MAXABS, TRUNC>(rc, g, M0, rr, wr);
    return;
  }
#endif
  switch (L) {
    case 0: warp_hier_top_L<0, MAXABS, TRUNC>(rc, g, M0, rr, scr, wr); break;
    case 1: warp_hier_top_L<1, MAXABS, TRUNC>(rc, g, M0, rr, scr, wr); break;
    case 2: warp_hier_top_L<2, MAXABS, TRUNC>(rc, g, M0, rr, scr, wr); break;
    default: warp_hier_top_L<3, MAXABS, TRUNC>(rc, g, M0, rr, scr, wr); break;
  }
}

// ------------------------------------------------------------------------------------------
// CTA-level sweep
// ------------------------------------------------------------------------------------------
constexpr int kMaxVerify = 32;  // candidates re-evaluated exactly after a hierarchical MAXABS sweep
#ifndef PP_FIRSTHIT_CHUNK
#define PP_FIRSTHIT_CHUNK 32
#endif
constexpr int kFirstHitChunk = PP_FIRSTHIT_CHUNK;  // candidates per speculation chunk of a first-hit sweep

struct SweepShared {
  double rcp[kRcpTab];  // rcp[m] = 1 / m (rcp[0] unused); filled once per CTA by sweep_shared_init
  SweepParams params;
  int counter;  // next candidate index
  int ncand;    // hierarchical MAXABS / fp32 nomination: candidates to verify
  unsigned long long stat_nominated, stat_fallback;  // fp32 nomination statistics (development aid)
  int cand[kMaxVerify];
  int hit_p;    // first-hit mode: lowest period over threshold so far
  int tie_count;  // near-tie audit: candidates inside the rounding bound of the best (1 = a clear winner)
  double wkey[kWarps];
  int wp[kWarps];
};

__device__ __forceinline__ void sweep_shared_init(SweepShared* sh) {
  if (threadIdx.x == 0) sh->stat_nominated = sh->stat_fallback = 0ull;
  for (int m = threadIdx.x; m < kRcpTab; m += kThreads) sh->rcp[m] = m ? 1.0 / (double)m : 0.0;
}

// Sweep all candidates with dynamic (atomic-counter) distribution over the CTA's warps.
//   argmax mode (thresh < 0): strict '>' from 0, lowest p on ties, periods in `skip` ignored
//                             (Periods.py:512-515).
//   first-hit mode (thresh >= 0): lowest p whose metric > thresh; warps stop once their next
//                             candidate lies above the current hit (Periods.py:273-286).
// sh->params must have been written by thread 0.  All threads call; the result is valid in all
// threads.  Contains CTA barriers.  Kept out of line so the caller's live state does not compete
// with the fold's registers.
// FEAT selects the ranking paths compiled into this instance (a kernel only carries the code it can reach):
constexpr int kSweepHier = 1;        // fp64 hierarchical NORM / GAMMA ranking
constexpr int kSweepHierMaxAbs = 2;  // hierarchical MAXABS nomination + exact verification
constexpr int kSweepF32 = 4;         // float nomination + exact verification
constexpr int kSweepPlain = 8;       // the caller never sweeps with trunc / orth / MAXABS / IMPOSED: energy folds only
constexpr int kSweepNoMetricOut = 16;  // the caller never asks for per-candidate metrics (drops the sqrt / divide of
                                       // key_to_value from every ranking site)
constexpr int kSweepTieAudit = 32;     // NORM / GAMMA argmax sweeps: exact re-ranking of near-tied candidates
constexpr int kSweepFirstHit = 64;     // first-hit (threshold) sweeps: small-to-large only
constexpr int kSweepHierTrunc = 128;   // hierarchical NORM / GAMMA ranking of truncated folds (trunc_to_integer_multiple)

// Rounding bound of a ranking key (an energy sum_r S_r^2 / cnt_r evaluated by any of the folds: sequential,
// hierarchical, reciprocal weights) against the exactly rounded one, relative to e >= sum x^2 of the swept signal:
// ceil(N/p) additions per residue, the squares, the reciprocal weights and the reductions (<= 40 u), doubled.
__device__ __forceinline__ double tie_tol(int N, int p, double e) {
  const double u = 1.1102230246251565e-16;  // 2^-53
  return 2.0 * (2.0 * (double)((N + p - 1) / p) + 40.0) * u * e;
}

// The reference's own evaluation of candidate p (Periods.py:504-510): the projection with sequential sums and IEEE
// means (bit-identical base vector), then the sum of squares of the tiled base over n < N in an order that does not
// depend on p -- so candidates with identical base vectors (p, 2p, 3p of an exactly periodic integer-valued input)
// tie EXACTLY, as they do in numpy.  Returns the ranking VALUE (norm, or gamma norm).  All threads call; barriers inside.
static __device__ __noinline__ double cta_canonical_value(const SweepParams* sp, SweepShared* sh, int p);
template <int FEAT>
static __device__ __noinline__ SweepResult cta_sweep(SweepShared* sh) {
  const SweepParams* sp = &sh->params;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    sh->counter = 0;
    sh->hit_p = 0x7fffffff;
  }
  __syncthreads();  // also publishes params written by thread 0 just before the call
  RankCtx rc_init = rank_ctx(sp);
  if constexpr ((FEAT & kSweepNoMetricOut) != 0) rc_init.metric_out = nullptr;
  const RankCtx rc = rc_init;
  const int metric = rc.metric;
  const int pmin = sp->pmin, pmax = sp->pmax;
  const double thresh = sp->thresh;
  const bool first_hit = (FEAT & kSweepFirstHit) != 0 && thresh >= 0.0;
  Best best{0.0, 0};
  // MAXABS (best-correlation) may rank hierarchically only when the caller provides `verify_keys`: the metric
  // must be the reference's bit-exact sequential sum, so the hierarchical pass only NOMINATES candidates and
  // the near-maximal ones are re-evaluated exactly below.
  const bool hier_maxabs = (FEAT & kSweepHierMaxAbs) != 0 && metric == PP_METRIC_MAXABS && sp->verify_keys != nullptr;
  const bool hier = (FEAT & (kSweepHier | kSweepHierMaxAbs | kSweepF32)) != 0 && sp->hier_scr != nullptr &&
                    sp->tops != nullptr && !first_hit && !sp->orth && (!sp->trunc || (FEAT & kSweepHierTrunc) != 0) &&
                    (((FEAT & (kSweepHier | kSweepF32)) != 0 && (metric == PP_METRIC_NORM || metric == PP_METRIC_GAMMA)) ||
                     hier_maxabs);
  // fp32 nomination: the float pass fills verify_keys[], then every candidate whose upper bound reaches the best
  // lower bound is folded sequentially in fp64 and ranked with the reference's rule.
  bool ranked = false;
  if constexpr ((FEAT & kSweepF32) != 0)
  if (hier && !hier_maxabs && sp->xf0_off != 0 && sp->verify_keys != nullptr && sp->metric_out == nullptr) {
    const uint2* __restrict__ tops = sp->tops;
    const int total = sp->ntops;
    double* scr = sp->hier_scr + (size_t)wid * sp->hier_len;
    double* keys = sp->verify_keys;
    const F32Window fw{sp->xf0_off, sp->xf1_off};
    double pend = 0.0;
    int pend_p = 0;
    while (true) {
      int idx = 0;
      if (lane == 0) idx = atomicAdd(&sh->counter, 1);
      idx = __shfl_sync(0xffffffffu, idx, 0);
      if (idx >= total) break;
      warp_hier_job_f32(rc, fw, keys, __ldg(tops + idx), scr, pend, pend_p);
    }
    if (pend_p != 0) {  // odd top left without a partner
      const double key = warp_sum(pend);
      if (lane == 0) keys[pend_p] = key;
    }
    if (threadIdx.x == 0) sh->ncand = 0;
    __syncthreads();  // every float energy is in keys[]
    const double e_res = sp->e_f32;
    const bool gam = metric == PP_METRIC_GAMMA;
    const uint32_t* skip = rc.skip;
    double lb = -1.0;  // best guaranteed lower bound of a ranking value
    for (int p = pmin + threadIdx.x; p <= pmax; p += kThreads) {
      if (skip != nullptr && ((skip[p >> 5] >> (p & 31)) & 1u)) continue;
      double v = keys[p] - f32_energy_tol(rc.N, p, e_res);
      if (gam) v = v / (double)p;
      lb = fmax(lb, v);
    }
    lb = warp_max(lb);
    if (lane == 0) sh->wkey[wid] = lb;
    __syncthreads();
    lb = sh->wkey[0];
#pragma unroll
    for (int w2 = 1; w2 < kWarps; ++w2) lb = fmax(lb, sh->wkey[w2]);
    for (int p = pmin + threadIdx.x; p <= pmax; p += kThreads) {
      if (skip != nullptr && ((skip[p >> 5] >> (p & 31)) & 1u)) continue;
      double v = keys[p] + f32_energy_tol(rc.N, p, e_res);
      if (gam) v = v / (double)p;
      if (v >= lb) {
        const int slot = atomicAdd(&sh->ncand, 1);
        if (slot < kMaxVerify) sh->cand[slot] = p;
      }
    }
    __syncthreads();
    const int nc = sh->ncand;
    if (threadIdx.x == 0) {
      sh->stat_nominated += (unsigned long long)nc;
      sh->stat_fallback += nc > kMaxVerify ? 1ull : 0ull;
    }
    if (rc.tie_keys != nullptr)   // near-tie audit: only the candidates verified below carry a key
      for (int p = pmin + threadIdx.x; p <= pmax; p += kThreads) rc.tie_keys[p] = 0.0;
    __syncthreads();
    if (nc <= kMaxVerify) {
      RankCtx vrc = rc;
      vrc.skip = nullptr;  // skipped periods were not nominated
      for (int c = wid; c < nc; c += kWarps) {
        const int p = sh->cand[c];
        consider(vrc, warp_period_key<kPassEnergy>(sp, p), p, best);
      }
      ranked = true;
    } else {  // too many near-ties for the float pass to separate: rank this sweep in fp64
      if (threadIdx.x == 0) sh->counter = 0;
    }
    __syncthreads();  // wkey is rewritten below
  }
  if (ranked) {
  } else if (hier) {
    // tops: candidates p with 2p > pmax; everything else is derived from exactly one of them
    const uint2* __restrict__ tops = sp->tops;
    const int total = sp->ntops;
    double* scr = sp->hier_scr + (size_t)wid * sp->hier_len;
    RankCtx hrc = rc;
    if (hier_maxabs) hrc.metric_out = sp->verify_keys;  // every candidate's hierarchical key, for the verification
    WarpRank wr{best, 0.0, 0};
    while (true) {
      int idx = 0;
      if (lane == 0) idx = atomicAdd(&sh->counter, 1);
      idx = __shfl_sync(0xffffffffu, idx, 0);
      if (idx >= total) break;
      const uint2 job = __ldg(tops + idx);
      if constexpr ((FEAT & kSweepHierMaxAbs) != 0) {
        if (hier_maxabs) warp_hier_top<true>(hrc, job, scr, wr);
      }
      if constexpr ((FEAT & kSweepHier) != 0) {
        if constexpr ((FEAT & kSweepHierTrunc) != 0) {
          if (!hier_maxabs && sp->trunc) warp_hier_top<false, true>(hrc, job, scr, wr);
        }
        if (!hier_maxabs && !sp->trunc) warp_hier_top<false>(hrc, job, scr, wr);
      }
    }
    if (wr.pend_p != 0)  // odd top left without a partner
      consider(hrc, hier_maxabs ? warp_max(wr.pend) : warp_sum(wr.pend), wr.pend_p, wr.best);
    best = warp_best(metric, wr.best);
  } else if (first_hit) {
    // First-hit mode walks the candidates in ascending chunks of kFirstHitChunk, every warp folding its share of a
    // chunk, and stops at the first chunk that holds a hit: the speculation past the hit is bounded by one chunk
    // (a free-running hand-out lets fast warps fold hundreds of candidates of a residual that is about to change
    // while one warp is still busy with the long rows of a small period; the kernel time then varied 7x run to run).
    for (int base = pmin; base <= pmax; base += kFirstHitChunk) {
      const int last = min(base + kFirstHitChunk - 1, pmax);
      for (int p = base + wid; p <= last; p += kWarps) {
        if (p > *reinterpret_cast<volatile int*>(&sh->hit_p)) break;
        const double key = (FEAT & kSweepPlain) != 0 ? warp_period_key<kPassEnergy>(sp, p) : warp_period_key_any(sp, p);
        if (rc.metric_out != nullptr && lane == 0) rc.metric_out[p] = key;
        if (key > thresh) {
          if (best.p == 0 || p < best.p) {
            best.p = p;
            best.key = key;
          }
          if (lane == 0) atomicMin(&sh->hit_p, p);
        }
      }
      __syncthreads();
      if (*reinterpret_cast<volatile int*>(&sh->hit_p) != 0x7fffffff) break;   // uniform: read behind the barrier
    }
  } else {
    const int ncand = pmax - pmin + 1;
    while (true) {
      int idx = 0;
      if (lane == 0) idx = atomicAdd(&sh->counter, 1);
      idx = __shfl_sync(0xffffffffu, idx, 0);
      if (idx >= ncand) break;
      const int p = pmin + idx;
      const double key = (FEAT & kSweepPlain) != 0 ? warp_period_key<kPassEnergy>(sp, p) : warp_period_key_any(sp, p);
      consider(rc, key, p, best);
    }
  }
  if (lane == 0) {
    sh->wkey[wid] = best.key;
    sh->wp[wid] = best.p;
  }
  __syncthreads();
  Best res{0.0, 0};
#pragma unroll
  for (int w = 0; w < kWarps; ++w) {
    const double k = sh->wkey[w];
    const int q = sh->wp[w];
    if (q == 0) continue;
    if (first_hit) {
      if (res.p == 0 || q < res.p) res = Best{k, q};
    } else if (better(metric, k, q, res)) {
      res = Best{k, q};
    }
  }
  if constexpr ((FEAT & kSweepHierMaxAbs) != 0)
  if (hier && hier_maxabs && res.p != 0) {
    // Exact verification.  A hierarchical sum differs from the sequential one by at most
    // err = 2 N eps sum|x| <= 2 N eps sqrt(N e_res); a candidate whose hierarchical key lies more than 2 err below
    // the hierarchical maximum cannot reach the exact maximum.  The others (normally just one) are folded
    // sequentially and ranked with the reference's rule (strict '>', lowest p on ties).
    const double err = 2.0 * (double)rc.N * 1.2e-16 * sqrt((double)rc.N * sp->e_res);
    const double floor_key = res.key - 2.0 * err - 1e-13 * res.key;
    const double* keys = sp->verify_keys;
    if (threadIdx.x == 0) sh->ncand = 0;
    __syncthreads();  // also: every key written during the sweep is visible
    for (int p = pmin + threadIdx.x; p <= pmax; p += kThreads) {
      if (keys[p] >= floor_key) {
        const int slot = atomicAdd(&sh->ncand, 1);
        if (slot < kMaxVerify) sh->cand[slot] = p;
      }
    }
    __syncthreads();
    const int nc = sh->ncand;
    Best exact{0.0, 0};
    if (nc <= kMaxVerify) {
      for (int c = wid; c < nc; c += kWarps) {
        const int p = sh->cand[c];
        consider(rc, warp_period_key<kPassMaxAbs>(sp, p), p, exact);
      }
    } else {  // degenerate input (masses of near-ties): fold every candidate sequentially
      for (int p = pmin + wid; p <= pmax; p += kWarps) consider(rc, warp_period_key<kPassMaxAbs>(sp, p), p, exact);
    }
    __syncthreads();  // wkey / wp were read by everyone above
    if (lane == 0) {
      sh->wkey[wid] = exact.key;
      sh->wp[wid] = exact.p;
    }
    __syncthreads();
    res = Best{0.0, 0};
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
      const double k = sh->wkey[w];
      const int q = sh->wp[w];
      if (q != 0 && better(metric, k, q, res)) res = Best{k, q};
    }
  }
  SweepResult out{0.0, res.p};
  if (res.p != 0) out.val = key_to_value(metric, res.key, res.p, rc.sqrtN);
  if constexpr ((FEAT & kSweepTieAudit) != 0) {
    if (!first_hit && sp->tie_keys != nullptr && (metric == PP_METRIC_NORM || metric == PP_METRIC_GAMMA)) {
      // Near-tie audit.  The keys above are energies rebuilt from reciprocal weights (and, hierarchically, from
      // derived sums): a few ulp from the reference's norm of the tiled base, which is enough to rank a multiple
      // of the true period above it when the input is exactly periodic.  Every candidate whose key can reach the
      // best one within the rounding bound is therefore re-evaluated the reference's way and ranked by VALUE with
      // strict '>' in ascending p (Periods.py:512-515).  On inputs with a noise floor exactly one candidate
      // qualifies and nothing is recomputed.
      int nnom = 0;
      if (res.p != 0) {
        const double* keys = sp->tie_keys;
        uint32_t* nom = sp->tie_nom;
        const int words = (pmax + 32) / 32;
        for (int i = threadIdx.x; i < words; i += kThreads) nom[i] = 0u;
        if (threadIdx.x == 0) sh->ncand = 0;
        __syncthreads();
        const double e_bound = sp->e_res;
        const bool gam = metric == PP_METRIC_GAMMA;
        const double lo_best = res.key - tie_tol(rc.N, res.p, e_bound);
        const uint32_t* skip = rc.skip;
        for (int p = pmin + threadIdx.x; p <= pmax; p += kThreads) {
          if (skip != nullptr && ((skip[p >> 5] >> (p & 31)) & 1u)) continue;
          const double hi = keys[p] + tie_tol(rc.N, p, e_bound);
          const bool in = gam ? hi * (double)res.p >= lo_best * (double)p : hi >= lo_best;
          if (in) {
            atomicOr(&nom[p >> 5], 1u << (p & 31));
            atomicAdd(&sh->ncand, 1);
          }
        }
        __syncthreads();
        nnom = sh->ncand;
        if (nnom > 1) {
          double best_v = 0.0;
          int best_p = 0;
          for (int wd = 0; wd < words; ++wd) {
            uint32_t bits = nom[wd];  // uniform
            while (bits) {
              const int p = wd * 32 + __ffs(bits) - 1;
              bits &= bits - 1;
              const double v = cta_canonical_value(sp, sh, p);
              if (v > best_v) {  // ascending p, strict '>': the lowest period keeps an exact tie
                best_v = v;
                best_p = p;
              }
            }
          }
          out.p = best_p;
          out.val = best_v;
        }
      }
      if (threadIdx.x == 0) sh->tie_count = nnom;
    }
  }
  __syncthreads();  // wkey/wp may be rewritten by the next sweep
  return out;
}

static __device__ __noinline__ double cta_canonical_value(const SweepParams* sp, SweepShared* sh, int p) {
  const int N = sp->N;
  const bool orth = sp->orth != 0;
  const int clen = orth ? sp->chain_off[p + 1] - sp->chain_off[p] : 0;
  __syncthreads();  // the scratch may still be read by the previous candidate's reduction
  cta_project_exact<false>(staged_window(), 0, N, p, sp->trunc != 0, orth ? sp->chain_q + sp->chain_off[p] : nullptr, clen,
                           sp->canon_v, sp->canon_u);
  const double* v = sp->canon_v;
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
  if ((threadIdx.x & 31) == 0) sh->wkey[threadIdx.x >> 5] = a;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < kWarps; ++w) t += sh->wkey[w];
  return key_to_value(sp->metric, t, p, sp->sqrtN);
}

}  // namespace pp
