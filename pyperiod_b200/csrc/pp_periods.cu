// pyperiod_b200 -- persistent on-chip kernels for the Sethares-Staley `Periods` algorithms
// (project, sweep, M-best / M-best-gamma, small-to-large, best-correlation) and their C ABI.
//
// One CTA owns one window at a time: the window is staged once into shared memory by a TMA
// bulk copy, every sweep / projection / residual update happens there, and only the compact
// periods / powers (and, on request, the bases) go back to HBM.  The grid is persistent:
// 2 CTAs per SM x SM count, windows handed out through a global counter (WindowQueue).
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include "../../include/pyperiod_b200.h"
#include "pp_common.cuh"
#include "pp_sweep.cuh"
#include "pp_host.cuh"

namespace pp {

// ------------------------------------------------------------------------------------------
// host-side error text
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
int fail(int code, const char* fmt, const char* a) {
  snprintf(g_err, sizeof(g_err), fmt, a);
  return code;
}
int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  return -100 - (int)e;
}

// ------------------------------------------------------------------------------------------
// shared-memory plan (identical on host and device)
// ------------------------------------------------------------------------------------------
struct SmemPlan {
  int xs_len;   // doubles: window + zero pad
  int pv;       // doubles: single-period vectors (vwin, utmp)
  int num;      // slots (M-best) / rounds
  int skip_words;
  int hier_len; // doubles per warp of hierarchical-sweep scratch (0 = none)
  int xf_len;   // floats per fp32 copy of the window (0 = none; two copies, see SweepParams::xf0)
  int tie_len;  // doubles of per-candidate ranking keys for the near-tie audit (0 = none)
  __host__ __device__ size_t off_vwin() const { return (size_t)xs_len * 8; }
  __host__ __device__ size_t off_utmp() const { return off_vwin() + (size_t)pv * 8; }
  // the hierarchical-sweep scratch is only live inside a sweep, vwin/utmp only between sweeps: they share bytes
  __host__ __device__ size_t off_hier() const { return off_vwin(); }
  // M-best step 2 also parks 32 doubles per warp at vwin (warp_slot_factor_norm): for max_length < 127 that is more
  // than two single-period vectors.  (Without this term warps 5..7 wrote into norms / fval behind the region: one
  // window in ~2 million came out with garbage powers at max_length = 64 -- found by a soak of the GPU suite.)
  __host__ __device__ size_t union_bytes() const {
    const size_t a = 2 * (size_t)pv * 8, b = (size_t)kWarps * hier_len * 8, c = (size_t)kWarps * 32 * 8;
    const size_t ab = a > b ? a : b;
    return ab > c ? ab : c;
  }
  __host__ __device__ size_t off_red() const { return off_vwin() + union_bytes(); }
  __host__ __device__ size_t off_norms() const { return off_red() + 2 * kWarps * 8; }
  __host__ __device__ size_t off_fval() const { return off_norms() + (size_t)((num + 1) & ~1) * 8; }
  __host__ __device__ size_t off_facs() const { return off_fval() + (size_t)kMaxFactors * 8; }
  __host__ __device__ size_t off_bar() const { return off_facs() + (size_t)kMaxFactors * 4; }
  __host__ __device__ size_t off_sweep() const { return off_bar() + 16; }
  __host__ __device__ size_t off_periods() const { return off_sweep() + ((sizeof(SweepShared) + 15) & ~15); }
  __host__ __device__ size_t off_slot() const { return off_periods() + (size_t)num * 4; }
  __host__ __device__ size_t off_skip() const { return off_slot() + (size_t)num * 4; }
  __host__ __device__ size_t off_misc() const { return off_skip() + (size_t)skip_words * 4; }
  __host__ __device__ size_t off_xf() const { return (off_misc() + 64 + 15) & ~(size_t)15; }
  __host__ __device__ size_t off_tie() const { return off_xf() + 2 * (size_t)xf_len * 4; }
  __host__ __device__ size_t off_nom() const { return off_tie() + (size_t)tie_len * 8; }
  __host__ __device__ size_t bytes() const { return off_nom() + (tie_len ? (size_t)skip_words * 4 : 0) + 16; }
};

// Floats after the window in the fp32 copies, all zero.  A masked tile of JR pair columns starting at ra < g reads
// the elements up to ra + 64 JR - 1 of each complete row, i.e. up to N + 64 JR - 2 in row M0 - 1 (the tail row only
// reads pairs that start below N).  The widest masked tile is half a top tile at L = 0: 4 pair columns, 256 floats.
constexpr int kF32Pad = 320;
static_assert(kF32Pad >= 64 * (hier_cols_f32<0>::value / 2) && kF32Pad >= 64,
              "the masked fp32 tiles must not read past the zero tail of the float copies");

__host__ __device__ inline SmemPlan make_plan(int N, int pmax, int num, bool sweep_pad, bool hier = false,
                                              bool f32 = false, bool tie = false) {
  SmemPlan pl;
  pl.tie_len = tie ? ((pmax + 2) & ~1) : 0;
  pl.hier_len = hier ? hier_scratch_len(pmax) : 0;
  pl.xf_len = (hier && f32) ? ((N + kF32Pad + 3) & ~3) : 0;
  pl.xs_len = sweep_pad ? ((N + kSweepPad + 1) & ~1) : ((N + 1) & ~1);
  pl.pv = (pmax + 2) & ~1;
  pl.num = num;
  pl.skip_words = (pmax + 32) / 32;
  return pl;
}

struct Smem {
  double* xs;
  double* vwin;
  double* utmp;
  double* red;
  double* norms;
  double* fval;
  int* facs;
  double* hier;
  uint64_t* bar;
  SweepShared* sweep;
  int* periods;
  int* slot;
  uint32_t* skip;
  int* misc;
  float* xf0;
  float* xf1;
  double* tie_keys;
  uint32_t* tie_nom;
  __device__ Smem(unsigned char* base, const SmemPlan& pl) {
    tie_keys = pl.tie_len ? reinterpret_cast<double*>(base + pl.off_tie()) : nullptr;
    tie_nom = pl.tie_len ? reinterpret_cast<uint32_t*>(base + pl.off_nom()) : nullptr;
    xs = reinterpret_cast<double*>(base);
    vwin = reinterpret_cast<double*>(base + pl.off_vwin());
    utmp = reinterpret_cast<double*>(base + pl.off_utmp());
    red = reinterpret_cast<double*>(base + pl.off_red());
    norms = reinterpret_cast<double*>(base + pl.off_norms());
    fval = reinterpret_cast<double*>(base + pl.off_fval());
    facs = reinterpret_cast<int*>(base + pl.off_facs());
    hier = pl.hier_len ? reinterpret_cast<double*>(base + pl.off_hier()) : nullptr;
    bar = reinterpret_cast<uint64_t*>(base + pl.off_bar());
    sweep = reinterpret_cast<SweepShared*>(base + pl.off_sweep());
    periods = reinterpret_cast<int*>(base + pl.off_periods());
    slot = reinterpret_cast<int*>(base + pl.off_slot());
    skip = reinterpret_cast<uint32_t*>(base + pl.off_skip());
    misc = reinterpret_cast<int*>(base + pl.off_misc());
    xf0 = pl.xf_len ? reinterpret_cast<float*>(base + pl.off_xf()) : nullptr;
    xf1 = pl.xf_len ? xf0 + pl.xf_len : nullptr;
  }
};

// fp32 copies of the (residual) window: xf0[n] = x[n], xf1[n] = x[n + 1]; zero past N.  No barrier inside.
__device__ __forceinline__ void refresh_f32_copies(const double* xs, int N, float* xf0, float* xf1) {
  for (int n = threadIdx.x; n < N; n += kThreads) {
    const float v = (float)xs[n];
    xf0[n] = v;
    if (n > 0) xf1[n - 1] = v;
  }
}

// e >= the sum of squares that cta_sum_sq rounded to `s` (N fma terms: relative error below N 2^-53)
__device__ __forceinline__ double f32_sum_sq_bound(double s, int N) { return fma(s, (double)(N + 2) * 0x1p-52, s); }

__device__ __forceinline__ void zero_pad(double* xs, int from, int to) {
  for (int i = from + threadIdx.x; i < to; i += kThreads) xs[i] = 0.0;
}

struct Tables {
  const int32_t* chain_off;
  const int32_t* chain_q;
  const int32_t* fac_off;
  const int32_t* fac;
};

// ------------------------------------------------------------------------------------------
// K0: Periods.project for a batch (Periods.py:142-219)
// ------------------------------------------------------------------------------------------
struct ChainArg {
  int32_t q[16];
  int32_t len;
};

__global__ void __launch_bounds__(kThreads, 2)
project_kernel(const double* __restrict__ x, int64_t ldx, int B, int N, int p, int trunc, ChainArg chain,
               double* __restrict__ out, int64_t ldo, int out_len) {
  unsigned char* smem_raw = pp_smem;
  const SmemPlan pl = make_plan(N, p, 0, false);
  Smem sm(smem_raw, pl);
  __shared__ int32_t s_chain[16];
  if (threadIdx.x < 16) s_chain[threadIdx.x] = chain.q[threadIdx.x];
  WindowLoader loader;
  loader.init(sm.bar);
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    loader.load(sm.xs, x + (size_t)b * ldx, N);
    cta_project_exact<false>(sm.xs, 0, N, p, trunc != 0, s_chain, chain.len, sm.vwin, sm.utmp);
    cta_store_tiled(out + (size_t)b * ldo, out_len, sm.vwin, p);
  }
}

// periodic_norm for a batch (Periods.py:221-241): out[b] = ||x_b|| / sqrt(N) [/ sqrt(p)]
__global__ void __launch_bounds__(kThreads)
norm_kernel(const double* __restrict__ x, int64_t ldx, int B, int N, int p, double* __restrict__ out) {
  __shared__ double red[kWarps];
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const double e = cta_sum_sq(x + (size_t)b * ldx, N, red);
    if (threadIdx.x == 0) {
      double v = sqrt(e) / sqrt((double)N);
      if (p > 0) v = v / sqrt((double)p);
      out[b] = v;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// K1: one sweep per window (parity probe and building block)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, kCtasPerSm)
sweep_kernel(const double* __restrict__ x, int64_t ldx, int B, int N, int pmin, int pmax, int metric, int trunc,
             int orth, int hier, Tables tb, double* __restrict__ metric_out, int32_t* __restrict__ best_p,
             double* __restrict__ best_val, double* __restrict__ warp_scr, const uint2* __restrict__ tops, int ntops, int* __restrict__ next_window) {
  unsigned char* smem_raw = pp_smem;
  const bool tie = metric == PP_METRIC_NORM || metric == PP_METRIC_GAMMA;
  const SmemPlan pl = make_plan(N, pmax, 0, true, hier != 0, false, tie);
  Smem sm(smem_raw, pl);
  WindowLoader loader;
  loader.init(sm.bar);
  zero_pad(sm.xs, N, pl.xs_len);
  sweep_shared_init(sm.sweep);
  for (WindowQueue wq(next_window); wq.b < B; wq.next()) {
    const int b = wq.b;
    loader.load(sm.xs, x + (size_t)b * ldx, N);
    double e_res = 0.0;
    if (metric == PP_METRIC_IMPOSED || tie) e_res = cta_sum_sq(sm.xs, N, sm.red);
    if (threadIdx.x == 0) {
      SweepParams& sp = sm.sweep->params;
      sp.N = N;
      sp.pmin = pmin;
      sp.pmax = pmax;
      sp.metric = metric;
      sp.trunc = trunc;
      sp.orth = orth;
      sp.chain_off = tb.chain_off;
      sp.chain_q = tb.chain_q;
      sp.warp_scr = warp_scr ? warp_scr + (size_t)blockIdx.x * kWarps * 2 * pl.pv : nullptr;
      sp.pv = pl.pv;
      sp.sqrtN = sqrt((double)N);
      sp.e_res = e_res;
      sp.data_norm = metric == PP_METRIC_IMPOSED ? sqrt(e_res) / sp.sqrtN : 1.0;
      sp.thresh = -1.0;
      sp.skip = nullptr;
      sp.nskip = 0;
      sp.hier_scr = sm.hier;
      sp.hier_len = pl.hier_len;
      sp.rcp = sm.sweep->rcp;
      sp.tops = tops;
      sp.ntops = ntops;
      sp.verify_keys = nullptr;
      sp.xf0_off = 0;
      sp.xf1_off = 0;
      sp.metric_out = metric_out ? metric_out + (size_t)b * (pmax + 1) : nullptr;
      sp.tie_keys = sm.tie_keys;
      sp.tie_nom = sm.tie_nom;
      sp.canon_v = sm.vwin;
      sp.canon_u = sm.utmp;
    }
    const SweepResult r = cta_sweep<kSweepHier | kSweepHierTrunc | kSweepTieAudit>(sm.sweep);
    if (threadIdx.x == 0) {
      best_p[b] = r.p;
      best_val[b] = r.val;
    }
  }
}

// ------------------------------------------------------------------------------------------
// K2: M-best / M-best-gamma, whole selection loop on chip (Periods.py:456-601)
// ------------------------------------------------------------------------------------------
// Norm of the projection of a P-periodic slot basis (tiled to N) onto a divisor f, by one warp.
// Ranking only (multiplicity sums instead of N sequential adds).
__device__ __forceinline__ double warp_slot_factor_norm(const double* slot, int P, int f, int N,
                                                        bool trunc, bool orth, const Tables& tb, double* scr,
                                                        double sqrtN, double* wscr) {
  // slot: the P-periodic basis (shared memory); wscr: 32 doubles of per-warp shared scratch
  const int lane = threadIdx.x & 31;
  const int t = P / f;
  const int Mf = N / f, r0f = N - Mf * f;
  // the mean of residue r divides by K_r in {Mf, Mf + 1}: two reciprocals instead of a division per residue
  const double rcp_lo = 1.0 / (double)Mf, rcp_hi = 1.0 / (double)(Mf + 1);
  double e = 0.0;
  if (f < 32) {
    // few residues, long sums: lane = (group, residue); the groups split the t terms of a residue and meet in
    // the scratch.  (One reduction per divisor: dependent shuffles queue behind the co-resident CTA's sweep.)
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
    warp_orth_chain_approx(scr, f, N, trunc, tb.chain_q + tb.chain_off[f], tb.chain_off[f + 1] - tb.chain_off[f]);
    for (int r = lane; r < f; r += 32) {
      const double v = scr[r];
      e = fma((double)(Mf + (r < r0f ? 1 : 0)) * v, v, e);
    }
    __syncwarp();
  }
  return sqrt(warp_sum(e)) / sqrtN;
}

// F32: the instance that carries the float-nomination sweep (PP_FOLD_NOMINATE_F32); the default instance does not
// (code that is compiled in but never reached still cost 3 % through layout and register allocation)
// PLAIN: neither trunc nor orth (the reference's default mode): those branches are compiled out.
template <bool F32, bool PLAIN>
__global__ void __launch_bounds__(kThreads, kCtasPerSm)
mbest_kernel(const double* __restrict__ x, int64_t ldx, int B, int N, int num, int pmin, int pmax, int gamma,
             int trunc_i, int orth_i, int hier, Tables tb, uint32_t* __restrict__ periods_out, double* __restrict__ powers_out,
             double* __restrict__ bases_out, int32_t* __restrict__ sweeps_out, int32_t* __restrict__ status_out,
             double* __restrict__ ws_slots, double* __restrict__ ws_scr, const uint2* __restrict__ tops, int ntops,
             int* __restrict__ next_window, unsigned long long* __restrict__ prof, int f32,
             int32_t* __restrict__ near_ties_out) {
  unsigned char* smem_raw = pp_smem;
  const SmemPlan pl = make_plan(N, pmax, num, true, hier != 0, f32 != 0, true);
  Smem sm(smem_raw, pl);
  const bool trunc = !PLAIN && trunc_i != 0, orth = !PLAIN && orth_i != 0;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const double sqrtN = sqrt((double)N);
  double* my_slots = ws_slots + (size_t)blockIdx.x * num * pl.pv;
  double* my_scr = ws_scr ? ws_scr + (size_t)blockIdx.x * kWarps * 2 * pl.pv : nullptr;
  // misc: [0]=filled [1]=repeats [2]=action [3]=slot storage id [4]=status [5]=step-2 decision [6]=chosen factor
  int* misc = sm.misc;

  WindowLoader loader;
  loader.init(sm.bar);
  zero_pad(sm.xs, N, pl.xs_len);
  sweep_shared_init(sm.sweep);
  if (sm.xf0 != nullptr) {  // zero tails of the fp32 copies (xf1[N-1] = x[N] = 0 included)
    for (int n = N - 1 + threadIdx.x; n < pl.xf_len; n += kThreads) {
      if (n >= N) sm.xf0[n] = 0.f;
      sm.xf1[n] = 0.f;
    }
  }

  // windows are handed out dynamically (global counter, zeroed per launch): per-window cost varies with the
  // number of sweeps and step-2 work, and a static stride leaves a tail of idle CTAs at the end of a launch
  int b = blockIdx.x;
  while (b < B) {
    int b_next = 0;
    if (threadIdx.x == 0) b_next = gridDim.x + atomicAdd(next_window, 1);  // consumed at the end of this window
    loader.load(sm.xs, x + (size_t)b * ldx, N);
    const double e_data = cta_sum_sq(sm.xs, N, sm.red);
    const double data_norm = sqrt(e_data) / sqrtN;  // periodic_norm(data), Periods.py:600
    // fp32 nomination only while no float value of a sweep can overflow: every residue sum and tile energy stays
    // below N sum x^2 (f32_energy_tol); other windows (and NaN / Inf data) rank with the fp64 hierarchy
    const bool f32_win = F32 && sm.xf0 != nullptr && (double)N * e_data <= 0x1p120;
    if (f32_win) refresh_f32_copies(sm.xs, N, sm.xf0, sm.xf1);  // published by the barrier below
    if (threadIdx.x == 0) {
      misc[0] = 0;
      misc[1] = 0;
      misc[4] = PP_STATUS_OK;
    }
    for (int i = threadIdx.x; i < num; i += kThreads) {
      sm.periods[i] = 0;
      sm.norms[i] = 0.0;
      sm.slot[i] = i;
    }
    for (int i = threadIdx.x; i < pl.skip_words; i += kThreads) sm.skip[i] = 0u;
    __syncthreads();

    if (threadIdx.x == 0) {
      SweepParams& sp = sm.sweep->params;
      sp.N = N;
      sp.pmin = pmin;
      sp.pmax = pmax;
      sp.metric = gamma ? PP_METRIC_GAMMA : PP_METRIC_NORM;
      sp.trunc = trunc;
      sp.orth = orth;
      sp.chain_off = tb.chain_off;
      sp.chain_q = tb.chain_q;
      sp.warp_scr = my_scr;
      sp.pv = pl.pv;
      sp.sqrtN = sqrtN;
      // bound of the near-tie audit: the residual of an orthogonal projection never has more energy than the data
      sp.e_res = e_data;
      sp.e_f32 = f32_sum_sq_bound(e_data, N);
      sp.data_norm = 1.0;
      sp.thresh = -1.0;
      sp.skip = sm.skip;
      sp.nskip = 0;
      sp.metric_out = nullptr;
      sp.hier_scr = sm.hier;
      sp.hier_len = pl.hier_len;
      sp.rcp = sm.sweep->rcp;
      sp.tops = tops;
      sp.ntops = ntops;
      // the float keys share the near-tie audit's key array: cta_sweep is done with them before the audit's keys
      // are written
      sp.verify_keys = f32_win ? sm.tie_keys : nullptr;
      sp.xf0_off = f32_win ? (int)pl.off_xf() : 0;
      sp.xf1_off = f32_win ? (int)(pl.off_xf() + (size_t)pl.xf_len * 4) : 0;
      sp.tie_keys = sm.tie_keys;
      sp.tie_nom = sm.tie_nom;
      sp.canon_v = sm.vwin;
      sp.canon_u = sm.utmp;
    }
    __syncthreads();

    // ---------------- step 1 (Periods.py:494-537)
    long long t_sweep = 0, t_proj = 0, t_upd = 0, t_step2 = 0, t_fac = 0, t_swap = 0, t_copy = 0, t_dec = 0, t_blk = 0, t_mark = clock64();
    int sweeps = 0, tie_sweeps = 0;
    const int guard = 12 * (pmax - pmin + 2) + 12 * num;
    while (true) {
      if (misc[0] >= num || misc[4] != PP_STATUS_OK) break;  // uniform: read after a barrier
      const SweepResult top = cta_sweep<kSweepHier | kSweepNoMetricOut | kSweepTieAudit | (F32 ? kSweepF32 : 0) |
                                        (PLAIN ? kSweepPlain : kSweepHierTrunc)>(sm.sweep);
      ++sweeps;
      if (sm.sweep->tie_count > 1) ++tie_sweeps;  // decided by the exact re-ranking
      { const long long t = clock64(); t_sweep += t - t_mark; t_mark = t; }
      if (top.p == 0 || sweeps > guard) {
        if (threadIdx.x == 0) misc[4] = top.p == 0 ? PP_STATUS_NO_PERIOD : PP_STATUS_GUARD;
        __syncthreads();
        break;
      }
      const int clen = orth ? tb.chain_off[top.p + 1] - tb.chain_off[top.p] : 0;
      cta_project_exact<false>(sm.xs, 0, N, top.p, trunc, orth ? tb.chain_q + tb.chain_off[top.p] : nullptr, clen,
                               sm.vwin, sm.utmp);
      { const long long t = clock64(); t_proj += t - t_mark; t_mark = t; }
      if (threadIdx.x == 0) {
        // (independent shared-memory loads issued as a batch: a lone thread's dependent loads queue behind
        // the other CTA's sweep traffic, ~200 cycles each)
        int found = -1;
        for (int i0 = 0; i0 < num; i0 += 16) {
          int pk[16];
#pragma unroll
          for (int k = 0; k < 16; ++k) pk[k] = (i0 + k < num) ? sm.periods[i0 + k] : -1;
#pragma unroll
          for (int k = 0; k < 16; ++k)
            if (pk[k] == top.p) found = i0 + k;
        }
        if (found >= 0 && misc[1] < 10) {          // strengthen an existing slot (:518-524)
          sm.norms[found] += top.val;
          misc[1] += 1;
          misc[2] = 0;
          misc[3] = sm.slot[found];
        } else if (found >= 0) {                   // blacklist it (:525-529)
          sm.skip[top.p >> 5] |= 1u << (top.p & 31);
          sm.sweep->params.nskip += 1;
          misc[1] = 0;
          misc[2] = 1;
        } else {                                   // new slot (:530-535)
          const int i = misc[0];
          sm.periods[i] = top.p;
          sm.norms[i] = top.val;
          misc[0] = i + 1;
          misc[1] = 0;
          misc[2] = 2;
          misc[3] = sm.slot[i];
        }
      }
      __syncthreads();
      const int action = misc[2];
      if (action != 1) {
        double* sl = my_slots + (size_t)misc[3] * pl.pv;
        if (action == 0) {
          for (int r = threadIdx.x; r < top.p; r += kThreads) sl[r] += sm.vwin[r];
        } else {
          for (int r = threadIdx.x; r < top.p; r += kThreads) sl[r] = sm.vwin[r];
        }
      }
      cta_subtract_tiled(sm.xs, N, sm.vwin, top.p);  // always (:537)
      if (f32_win) {
        __syncthreads();
        refresh_f32_copies(sm.xs, N, sm.xf0, sm.xf1);
        // the next sweep's float error scales with the residual's energy, which falls round by round
        const double e_now = cta_sum_sq(sm.xs, N, sm.red);
        if (threadIdx.x == 0) sm.sweep->params.e_f32 = f32_sum_sq_bound(e_now, N);
      }
      __syncthreads();
      { const long long t = clock64(); t_upd += t - t_mark; t_mark = t; }
    }

    // ---------------- step 2 (Periods.py:540-598), one pass
    int changes_total = 0;
    if (misc[4] == PP_STATUS_OK) {
      const double stale_div = sqrt((double)pmax);  // gamma norms divide by sqrt(max_length) (:559,:572)
      int i = 0;
      int changes = 0;
      while (i < num) {
        const int P = sm.periods[i];
        const double* sl = my_slots + (size_t)sm.slot[i] * pl.pv;
        const int f0 = tb.fac_off[P], nf = tb.fac_off[P + 1] - f0;
        if (nf > kMaxFactors || changes > 64 * num) {
          if (threadIdx.x == 0) misc[4] = PP_STATUS_GUARD;
          __syncthreads();
          break;
        }
        // the residual is dead after step 1: stage the slot basis (one period) and its divisor list on chip
        double* sl_s = sm.xs;
        const long long t_c0 = clock64();
        for (int r = threadIdx.x; r < P; r += kThreads) sl_s[r] = sl[r];
        for (int fi = threadIdx.x; fi < nf; fi += kThreads) sm.facs[fi] = tb.fac[f0 + fi];
        __syncthreads();
        const long long t_f0 = clock64();
        t_copy += t_f0 - t_c0;
        // every warp ranks its own divisors (ascending fi, strict '>' keeps the first maximum, Periods.py:561-565)
        double w_top = 0.0;
        int w_fi = -1;
        for (int fi = wid; fi < nf; fi += kWarps) {
          const int f = sm.facs[fi];
          double v = warp_slot_factor_norm(sl_s, P, f, N, trunc, orth, tb, my_scr ? my_scr + (size_t)wid * 2 * pl.pv : nullptr,
                                           sqrtN, sm.vwin + wid * 32);
          if (gamma) v = v / stale_div;
          if (v > w_top) {
            w_top = v;
            w_fi = fi;
          }
          if (fi == nf - 1 && lane == 0) sm.fval[0] = v;  // norm of the LAST factor's projection (:570-572)
        }
        if (lane == 0) {
          sm.sweep->wkey[wid] = w_top;
          sm.sweep->wp[wid] = w_fi;
        }
        __syncthreads();
        t_fac += clock64() - t_f0;
        if (threadIdx.x == 0) {
          const long long t_b0 = clock64();
          double top = 0.0;
          int top_fi = -1;
          {
            double wk[kWarps];
            int wf[kWarps];
#pragma unroll
            for (int w = 0; w < kWarps; ++w) {
              wk[w] = sm.sweep->wkey[w];
              wf[w] = sm.sweep->wp[w];
            }
#pragma unroll
            for (int w = 0; w < kWarps; ++w)
              if (wf[w] >= 0 && (wk[w] > top || (wk[w] == top && top_fi >= 0 && wf[w] < top_fi))) {
                top = wk[w];
                top_fi = wf[w];
              }
          }
          const int top_f = top_fi >= 0 ? sm.facs[top_fi] : 0;
          int decision = 0;
          if (top_f != 0) {
            bool present = false;
            double floor_n = sm.norms[0];
            const double n_weak = sm.fval[0], n_last = sm.norms[num - 1], n_i = sm.norms[i];
            for (int k0 = 0; k0 < num; k0 += 16) {  // batched loads, see step 1
              int pk[16];
              double nk[16];
#pragma unroll
              for (int k = 0; k < 16; ++k) {
                pk[k] = (k0 + k < num) ? sm.periods[k0 + k] : -1;
                nk[k] = (k0 + k < num) ? sm.norms[k0 + k] : floor_n;
              }
#pragma unroll
              for (int k = 0; k < 16; ++k) {
                present |= (pk[k] == top_f);
                if (k0 + k < num) floor_n = fmin(floor_n, nk[k]);
              }
            }
            if (!present) {
              const double n_strong = top;
              if ((n_weak + n_strong) > (n_last + n_i) && n_weak > floor_n && n_strong > floor_n) {
                decision = 1;
                // slot i keeps its period with the weakened basis; the strong factor is inserted before it
                const int freed = sm.slot[num - 1];
                for (int k = num - 1; k > i; --k) {
                  sm.periods[k] = sm.periods[k - 1];
                  sm.norms[k] = sm.norms[k - 1];
                  sm.slot[k] = sm.slot[k - 1];
                }
                // after the shift, entries i and i+1 both describe the old slot (when i+1 < num)
                if (i + 1 < num) sm.norms[i + 1] = n_weak;
                sm.periods[i] = top_f;
                sm.norms[i] = n_strong;
                sm.slot[i] = freed;
                misc[3] = freed;
              }
            }
          }
          misc[5] = decision;
          misc[6] = top_f;
          t_blk += clock64() - t_b0;
        }
        __syncthreads();
        t_dec += clock64() - t_f0;
        if (misc[5]) {
          const long long t_s0 = clock64();
          const int f = misc[6];
          const int clen = orth ? tb.chain_off[f + 1] - tb.chain_off[f] : 0;
          // exact xQ = project(bases[i], f) from the (still unmodified) old slot storage
          cta_project_exact<true>(sl_s, P, N, f, trunc, orth ? tb.chain_q + tb.chain_off[f] : nullptr, clen, sm.vwin,
                                  sm.utmp);
          double* old_sl = const_cast<double*>(sl);
          double* new_sl = my_slots + (size_t)misc[3] * pl.pv;
          const bool old_survives = (i + 1 < num);
          // xq = bases[i] - xQ (elementwise on one period), unless the old slot was the one dropped
          if (old_survives) {
            int rq = threadIdx.x % f;
            const int step = kThreads % f;
            for (int r = threadIdx.x; r < P; r += kThreads) {
              old_sl[r] = sl_s[r] - sm.vwin[rq];
              rq += step;
              if (rq >= f) rq -= f;
            }
          }
          __syncthreads();  // old_sl may alias new_sl when the old slot was dropped
          for (int r = threadIdx.x; r < f; r += kThreads) new_sl[r] = sm.vwin[r];
          ++changes;
          ++changes_total;
          __syncthreads();
          t_swap += clock64() - t_s0;
        } else {
          ++i;
        }
      }
    }

    // ---------------- outputs
    __syncthreads();
    t_step2 = clock64() - t_mark;
    if (prof != nullptr && threadIdx.x == 0) {
      atomicAdd(prof + 0, (unsigned long long)t_sweep);
      atomicAdd(prof + 1, (unsigned long long)t_proj);
      atomicAdd(prof + 2, (unsigned long long)t_upd);
      atomicAdd(prof + 3, (unsigned long long)t_step2);
      atomicAdd(prof + 4, 1ull);
      atomicAdd(prof + 5, (unsigned long long)t_fac);
      if (sm.xf0 != nullptr) {  // fp32 nomination statistics instead of the step-2 detail
        atomicAdd(prof + 6, sm.sweep->stat_nominated);
        atomicAdd(prof + 7, sm.sweep->stat_fallback);
        sm.sweep->stat_nominated = sm.sweep->stat_fallback = 0ull;
      } else {
        atomicAdd(prof + 6, (unsigned long long)t_dec);
        atomicAdd(prof + 7, (unsigned long long)t_blk);
      }
    }
    const int status = misc[4];
    for (int i = threadIdx.x; i < num; i += kThreads) {
      const bool ok = status == PP_STATUS_OK;
      periods_out[(size_t)b * num + i] = ok ? (uint32_t)sm.periods[i] : 0u;
      powers_out[(size_t)b * num + i] = ok ? sm.norms[i] / data_norm : 0.0;
    }
    if (threadIdx.x == 0) {
      status_out[b] = status;
      if (sweeps_out) sweeps_out[b] = sweeps;
      if (near_ties_out) near_ties_out[b] = tie_sweeps;
    }
    if (bases_out != nullptr) {
      for (int i = 0; i < num; ++i) {
        double* dst = bases_out + ((size_t)b * num + i) * N;
        const int P = sm.periods[i];
        if (status == PP_STATUS_OK && P > 0) {
          // the residual is dead: stage the one-period basis in shared memory, then stream its tiling out
          const double* sl = my_slots + (size_t)sm.slot[i] * pl.pv;
          __syncthreads();
          for (int r = threadIdx.x; r < P; r += kThreads) sm.xs[r] = sl[r];
          __syncthreads();
          cta_store_tiled(dst, N, sm.xs, P);
        } else {
          for (int n = threadIdx.x; n < N; n += kThreads) __stcs(dst + n, 0.0);
        }
      }
    }
    if (threadIdx.x == 0) misc[7] = b_next;
    __syncthreads();
    b = misc[7];
  }
}

// ------------------------------------------------------------------------------------------
// K3: small-to-large (Periods.py:246-287): speculative sweep, restart after each acceptance
// ------------------------------------------------------------------------------------------
// small-to-large is a chain of short phases (a few candidates between restarts, projection, update): latency bound,
// so a third CTA per SM pays (17.1 vs 20.8 ms for 16,384 windows of N = 2048; 80 registers, no spills)
constexpr int kS2lCtasPerSm = 3;

__global__ void __launch_bounds__(kThreads, kS2lCtasPerSm)
s2l_kernel(const double* __restrict__ x, int64_t ldx, int B, int N, double thresh, int n_periods, int trunc_i,
           int orth_i, Tables tb, int kmax, uint32_t* __restrict__ periods_out, double* __restrict__ powers_out,
           double* __restrict__ bases_out, int32_t* __restrict__ count_out, int32_t* __restrict__ status_out,
           double* __restrict__ ws_scr, int* __restrict__ next_window) {
  unsigned char* smem_raw = pp_smem;
  const SmemPlan pl = make_plan(N, n_periods, 0, true);
  Smem sm(smem_raw, pl);
  const bool trunc = trunc_i != 0, orth = orth_i != 0;
  const double sqrtN = sqrt((double)N);
  double* my_scr = ws_scr ? ws_scr + (size_t)blockIdx.x * kWarps * 2 * pl.pv : nullptr;
  WindowLoader loader;
  loader.init(sm.bar);
  zero_pad(sm.xs, N, pl.xs_len);
  sweep_shared_init(sm.sweep);
  for (WindowQueue wq(next_window); wq.b < B; wq.next()) {
    const int b = wq.b;
    loader.load(sm.xs, x + (size_t)b * ldx, N);
    const double e_data = cta_sum_sq(sm.xs, N, sm.red);
    if (threadIdx.x == 0) {
      SweepParams& sp = sm.sweep->params;
      sp.N = N;
      sp.pmax = n_periods;
      sp.metric = PP_METRIC_IMPOSED;
      sp.trunc = trunc;
      sp.orth = orth;
      sp.chain_off = tb.chain_off;
      sp.chain_q = tb.chain_q;
      sp.warp_scr = my_scr;
      sp.pv = pl.pv;
      sp.sqrtN = sqrtN;
      sp.e_res = e_data;
      sp.data_norm = sqrt(e_data) / sqrtN;
      sp.thresh = thresh < 0.0 ? 0.0 : thresh;
      sp.skip = nullptr;
      sp.nskip = 0;
      sp.metric_out = nullptr;
      sp.hier_scr = nullptr;
      sp.hier_len = 0;
      sp.rcp = sm.sweep->rcp;
      sp.tops = nullptr;
      sp.ntops = 0;
      sp.verify_keys = nullptr;
      sp.xf0_off = 0;
      sp.xf1_off = 0;
      sp.tie_keys = nullptr;
      sp.tie_nom = nullptr;
      sp.canon_v = nullptr;
      sp.canon_u = nullptr;
    }
    int count = 0;
    int pstart = 2;
    // thresh < 0 would accept every period in the reference; first-hit mode needs thresh >= 0,
    // the host rejects negative thresholds.
    while (pstart <= n_periods) {
      if (threadIdx.x == 0) sm.sweep->params.pmin = pstart;
      const SweepResult hit = cta_sweep<kSweepFirstHit>(sm.sweep);
      if (hit.p == 0) break;
      const int clen = orth ? tb.chain_off[hit.p + 1] - tb.chain_off[hit.p] : 0;
      cta_project_exact<false>(sm.xs, 0, N, hit.p, trunc, orth ? tb.chain_q + tb.chain_off[hit.p] : nullptr, clen,
                               sm.vwin, sm.utmp);
      cta_subtract_tiled(sm.xs, N, sm.vwin, hit.p);
      if (count < kmax) {
        if (threadIdx.x == 0) {
          periods_out[(size_t)b * kmax + count] = (uint32_t)hit.p;
          powers_out[(size_t)b * kmax + count] = hit.val;
        }
        if (bases_out) cta_store_tiled(bases_out + ((size_t)b * kmax + count) * N, N, sm.vwin, hit.p);
      }
      ++count;
      __syncthreads();
      const double e_now = cta_sum_sq(sm.xs, N, sm.red);
      if (threadIdx.x == 0) sm.sweep->params.e_res = e_now;
      pstart = hit.p + 1;
    }
    for (int k = count + threadIdx.x; k < kmax; k += kThreads) {
      periods_out[(size_t)b * kmax + k] = 0u;
      powers_out[(size_t)b * kmax + k] = 0.0;
    }
    if (threadIdx.x == 0) {
      count_out[b] = count;
      status_out[b] = count > kmax ? PP_STATUS_OVERFLOW : PP_STATUS_OK;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// K4: best-correlation (Periods.py:289-349)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, kCtasPerSm)
bcorr_kernel(const double* __restrict__ x, int64_t ldx, int B, int N, int num, int max_length, double ratio,
             int trunc_i, int orth_i, Tables tb, uint32_t* __restrict__ periods_out, double* __restrict__ powers_out,
             double* __restrict__ bases_out, int32_t* __restrict__ status_out, int* __restrict__ next_window,
             int hier, double* __restrict__ ws_keys, const uint2* __restrict__ tops, int ntops) {
  unsigned char* smem_raw = pp_smem;
  const SmemPlan pl = make_plan(N, max_length, 0, true, hier != 0);
  Smem sm(smem_raw, pl);
  const bool trunc = trunc_i != 0, orth = orth_i != 0;
  const double sqrtN = sqrt((double)N);
  WindowLoader loader;
  loader.init(sm.bar);
  zero_pad(sm.xs, N, pl.xs_len);
  sweep_shared_init(sm.sweep);
  for (WindowQueue wq(next_window); wq.b < B; wq.next()) {
    const int b = wq.b;
    loader.load(sm.xs, x + (size_t)b * ldx, N);
    double e_now = cta_sum_sq(sm.xs, N, sm.red);   // sum x^2 of the current residual
    const double og = sqrt(e_now) / sqrtN;
    double prev = og;
    int status = PP_STATUS_OK;
    if (threadIdx.x == 0) {
      SweepParams& sp = sm.sweep->params;
      sp.N = N;
      sp.pmin = 2;
      sp.pmax = max_length - 1;  // range(2, max_length) excludes max_length (:324)
      sp.metric = PP_METRIC_MAXABS;
      sp.trunc = 0;              // the correlation metric always folds all N samples
      sp.orth = 0;
      sp.chain_off = tb.chain_off;
      sp.chain_q = tb.chain_q;
      sp.warp_scr = nullptr;
      sp.pv = pl.pv;
      sp.sqrtN = sqrtN;
      sp.e_res = 0.0;
      sp.data_norm = 1.0;
      sp.thresh = -1.0;
      sp.skip = nullptr;
      sp.nskip = 0;
      sp.metric_out = nullptr;
      // hierarchical MAXABS ranking + exact verification of the near-maximal candidates (pp_sweep.cuh)
      sp.hier_scr = hier ? sm.hier : nullptr;
      sp.hier_len = pl.hier_len;
      sp.rcp = sm.sweep->rcp;
      sp.tops = tops;
      sp.ntops = ntops;
      sp.verify_keys = hier ? ws_keys + (size_t)blockIdx.x * (max_length + 1) : nullptr;
      sp.xf0_off = 0;
      sp.xf1_off = 0;
      sp.tie_keys = nullptr;
      sp.tie_nom = nullptr;
      sp.canon_v = nullptr;
      sp.canon_u = nullptr;
    }
    for (int i = 0; i < num; ++i) {
      uint32_t out_p = 0u;
      double out_v = 0.0;
      bool keep = false;
      int p_sel = 0;
      if (status == PP_STATUS_OK) {
        if (threadIdx.x == 0) sm.sweep->params.e_res = e_now;  // error bound of the hierarchical sums
        const SweepResult top = cta_sweep<kSweepHierMaxAbs>(sm.sweep);
        if (top.p == 0) {
          status = PP_STATUS_NO_PERIOD;
        } else {
          p_sel = top.p;
          const int clen = orth ? tb.chain_off[top.p + 1] - tb.chain_off[top.p] : 0;
          cta_project_exact<false>(sm.xs, 0, N, top.p, trunc, orth ? tb.chain_q + tb.chain_off[top.p] : nullptr, clen,
                                   sm.vwin, sm.utmp);
          cta_subtract_tiled(sm.xs, N, sm.vwin, top.p);  // always (:340)
          __syncthreads();
          e_now = cta_sum_sq(sm.xs, N, sm.red);
          const double now = sqrt(e_now) / sqrtN;
          const double drop = (prev - now) / og;
          if (drop > ratio) {
            keep = true;
            out_p = (uint32_t)top.p;
            out_v = drop;
            prev = now;
          }
        }
      }
      if (threadIdx.x == 0) {
        periods_out[(size_t)b * num + i] = out_p;
        powers_out[(size_t)b * num + i] = out_v;
      }
      if (bases_out) {
        double* dst = bases_out + ((size_t)b * num + i) * N;
        if (keep) cta_store_tiled(dst, N, sm.vwin, p_sel);
        else
          for (int n = threadIdx.x; n < N; n += kThreads) __stcs(dst + n, 0.0);
      }
      __syncthreads();
    }
    if (threadIdx.x == 0) status_out[b] = status;
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
// hierarchical ranking sweeps where they apply, unless the call asks for direct folds
// (orthogonalised sweeps need every candidate's projection vector, not just its energy: sequential folds).  Truncated
// folds (trunc_to_integer_multiple) rank hierarchically too (never in float).
static bool hier_applies(int fold_mode, int metric, int trunc, int orth) {
  (void)trunc;
  return fold_mode != PP_FOLD_DIRECT && !orth && (metric == PP_METRIC_NORM || metric == PP_METRIC_GAMMA);
}
static bool hier_riders(int fold_mode, int trunc) {
  (void)trunc;   // truncated folds ride too (the same top-set correction applies to the 3 * 2^i set arrays)
  return fold_mode != PP_FOLD_HIERARCHICAL_NO_RIDERS;
}

// plan used for grid / workspace sizing: the largest any fold mode of the algorithm needs
static int plan_for(int algo, int N, int pmax, int num, SmemPlan& pl) {
  pl = make_plan(N, pmax, algo == PP_ALGO_MBEST ? num : 0, true, algo == PP_ALGO_MBEST || algo == PP_ALGO_SWEEP || algo == PP_ALGO_BCORR,
                 false, algo == PP_ALGO_MBEST || algo == PP_ALGO_SWEEP);
  return 0;
}

}  // namespace pp

using namespace pp;

extern "C" {

int pp_abi_version(void) { return PP_ABI_VERSION; }

int pp_sweep_passes(int32_t N, int32_t pmin, int32_t pmax, int32_t fold_mode) {
  if (pmax < pmin) return 0;
  if (fold_mode == PP_FOLD_DIRECT) return pmax - pmin + 1;
  return hier_job_count(N, pmin, pmax, fold_mode != PP_FOLD_HIERARCHICAL_NO_RIDERS);
}
const char* pp_last_error(void) { return g_err; }

int pp_device_info(int32_t* sm_count, int32_t* smem_optin_bytes, int32_t* cc_major, int32_t* cc_minor,
                   int32_t* clock_khz) {
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  if (sm_count) *sm_count = f.sm_count;
  if (smem_optin_bytes) *smem_optin_bytes = f.smem_optin;
  if (cc_major) *cc_major = f.major;
  if (cc_minor) *cc_minor = f.minor;
  if (clock_khz) *clock_khz = f.clock_khz;
  return 0;
}

int pp_grid_size(int32_t algo, int32_t N, int32_t pmax, int32_t orth) {
  (void)orth;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  SmemPlan pl;
  plan_for(algo, N, pmax, 16, pl);
  return grid_for(f, pl.bytes(), 0, algo == PP_ALGO_S2L ? kS2lCtasPerSm : kCtasPerSm);
}

size_t pp_workspace_bytes(int32_t algo, int32_t N, int32_t pmax, int32_t num, int32_t orth) {
  DeviceFacts f;
  if (device_facts(f)) return 0;
  SmemPlan pl;
  plan_for(algo, N, pmax, num, pl);
  // upper bound on the persistent grid
  const size_t grid = (size_t)f.sm_count * (algo == PP_ALGO_S2L ? kS2lCtasPerSm : kCtasPerSm);
  size_t bytes = 1024 + 1024 + (size_t)(pmax + 2) * sizeof(uint2);
  if (algo == PP_ALGO_MBEST) bytes += grid * (size_t)num * pl.pv * 8;
  if (orth && algo != PP_ALGO_BCORR) bytes += grid * kWarps * 2 * (size_t)pl.pv * 8;
  if (algo == PP_ALGO_BCORR) bytes += grid * (size_t)(pmax + 2) * 8;  // hierarchical keys awaiting verification
  return bytes;
}

int pp_fits_on_chip(int32_t algo, int32_t N, int32_t pmax, int32_t num, int32_t metric, int32_t trunc, int32_t orth,
                    int32_t fold_mode, int32_t smem_bytes) {
  if (N < 1 || pmax < 0 || num < 0 || metric < 0 || metric > 3 || smem_bytes < 0) return fail(-1, "bad arguments%s");
  if (check_fold_mode(fold_mode)) return -1;
  size_t bytes = 0;
  switch (algo) {
    case PP_ALGO_PROJECT: bytes = make_plan(N, pmax, 0, false).bytes(); break;
    case PP_ALGO_SWEEP:
      bytes = make_plan(N, pmax, 0, true, hier_applies(fold_mode, metric, trunc, orth), false,
                        metric == PP_METRIC_NORM || metric == PP_METRIC_GAMMA).bytes();
      break;
    case PP_ALGO_MBEST: {
      const bool hier = hier_applies(fold_mode, metric, trunc, orth);
      bytes = make_plan(N, pmax, num, true, hier, hier && !trunc && fold_mode == PP_FOLD_NOMINATE_F32, true).bytes();
      break;
    }
    case PP_ALGO_S2L: bytes = make_plan(N, pmax, 0, true).bytes(); break;
    case PP_ALGO_BCORR:
      bytes = make_plan(N, pmax, 0, true, fold_mode != PP_FOLD_DIRECT && pmax - 1 >= 4).bytes();
      break;
    case PP_ALGO_BFREQ: bytes = bfreq_smem_bytes(N); break;
    default: return fail(-1, "unknown algorithm%s");
  }
  return bytes <= (size_t)smem_bytes ? 1 : 0;
}

static int check_common(const void* x, int64_t ldx, int B, int N) {
  if (x == nullptr) return fail(-1, "x is null%s");
  if (B < 0 || N < 2) return fail(-1, "need B >= 0 and N >= 2%s");
  if (ldx < 1) return fail(-1, "ldx must be >= 1%s");
  return 0;
}

int pp_project(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t p, int32_t trunc,
               const int32_t* chain_q_host, int32_t chain_len, double* out, int64_t ldo, int32_t out_len,
               void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (int rc = check_common(x, ldx, B, N)) return rc;
  if (p < 1 || p > N) return fail(-1, "period must satisfy 1 <= p <= N%s");
  if (chain_len < 0 || chain_len > 16) return fail(-1, "chain_len must be in [0,16]%s");
  if (out == nullptr || out_len < 1 || out_len > N || ldo < out_len) return fail(-1, "bad output shape%s");
  if (B == 0) return 0;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  const SmemPlan pl = make_plan(N, p, 0, false);
  if (int rc = prep_kernel(project_kernel, pl.bytes(), f)) return rc;
  ChainArg ca;
  memset(&ca, 0, sizeof(ca));
  ca.len = chain_len;
  for (int i = 0; i < chain_len; ++i) {
    if (chain_q_host[i] < 1 || chain_q_host[i] >= p || p % chain_q_host[i]) return fail(-1, "chain cofactor must divide p%s");
    ca.q[i] = chain_q_host[i];
  }
  project_kernel<<<grid_for(f, pl.bytes(), B), kThreads, pl.bytes(), (cudaStream_t)stream>>>(x, ldx, B, N, p, trunc, ca,
                                                                                            out, ldo, out_len);
  return check_cuda(cudaGetLastError(), "project_kernel launch");
}

int pp_periodic_norm(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t p, double* out, void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (x == nullptr || out == nullptr || B < 0 || N < 1 || ldx < 1 || p < 0) return fail(-1, "bad arguments%s");
  if (B == 0) return 0;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  int grid = f.sm_count * 4;
  if (grid > B) grid = B;
  norm_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(x, ldx, B, N, p, out);
  return check_cuda(cudaGetLastError(), "norm_kernel launch");
}

int pp_sweep(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t pmin, int32_t pmax, int32_t metric,
             int32_t trunc, int32_t orth, int32_t fold_mode, const int32_t* chain_off, const int32_t* chain_q,
             int32_t table_pmax, double* metric_out, int32_t* best_p, double* best_val, void* workspace,
             size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (int rc = check_common(x, ldx, B, N)) return rc;
  if (pmin < 1 || pmax < pmin || pmax > N) return fail(-1, "need 1 <= pmin <= pmax <= N%s");
  if (metric < 0 || metric > 3) return fail(-1, "unknown metric%s");
  if (metric == PP_METRIC_MAXABS && (trunc || orth)) return fail(-1, "MAXABS ignores trunc/orth; pass 0%s");
  if (orth && (chain_off == nullptr || chain_q == nullptr || table_pmax < pmax)) return fail(-1, "orth needs tables covering pmax%s");
  if (best_p == nullptr || best_val == nullptr) return fail(-1, "best_p/best_val are null%s");
  if (int rc = check_fold_mode(fold_mode)) return rc;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  const int hier = hier_applies(fold_mode, metric, trunc, orth) ? 1 : 0;
  const SmemPlan pl = make_plan(N, pmax, 0, true, hier != 0, false, metric == PP_METRIC_NORM || metric == PP_METRIC_GAMMA);
  if (int rc = prep_kernel(sweep_kernel, pl.bytes(), f)) return rc;
  const int grid = grid_for(f, pl.bytes(), B);
  size_t off = 0;
  double* scr = nullptr;
  if (orth) {
    scr = carve(workspace, workspace_bytes, off, (size_t)grid * kWarps * 2 * pl.pv * 8);
    if (!scr) return fail(-3, "workspace too small (see pp_workspace_bytes)%s");
  }
  uint2* tops = nullptr;
  int ntops = hier ? hier_top_count(pmin, pmax) : 0;
  if (ntops > 0) {
    tops = reinterpret_cast<uint2*>(carve(workspace, workspace_bytes, off, (size_t)ntops * sizeof(uint2)));
    if (!tops) return fail(-3, "workspace too small (see pp_workspace_bytes)%s");
    ntops = build_hier_jobs(N, pmin, pmax, hier_riders(fold_mode, trunc), tops, (cudaStream_t)stream);
  }
  Tables tb{chain_off, chain_q, nullptr, nullptr};
  int* next_window = carve_window_counter(workspace, workspace_bytes, off, (cudaStream_t)stream);
  sweep_kernel<<<grid, kThreads, pl.bytes(), (cudaStream_t)stream>>>(x, ldx, B, N, pmin, pmax, metric, trunc, orth, hier,
                                                                     tb, metric_out, best_p, best_val, scr, tops, ntops,
                                                                     next_window);
  return check_cuda(cudaGetLastError(), "sweep_kernel launch");
}

int pp_mbest(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t num, int32_t pmin, int32_t pmax,
             int32_t gamma, int32_t trunc, int32_t orth, int32_t fold_mode, const int32_t* chain_off,
             const int32_t* chain_q, const int32_t* fac_off, const int32_t* fac, int32_t table_pmax, uint32_t* periods,
             double* powers, double* bases, int32_t* sweeps, int32_t* near_ties, int32_t* status, void* workspace,
             size_t workspace_bytes, void* profile, void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (int rc = check_common(x, ldx, B, N)) return rc;
  if (num < 1 || num > 4096) return fail(-1, "need 1 <= num <= 4096%s");
  if (pmin < 2 || pmax < pmin || pmax > N) return fail(-1, "need 2 <= pmin <= pmax <= N%s");
  if (pmax - pmin + 1 < num) return fail(-1, "fewer candidate periods than num%s");
  if (fac_off == nullptr || fac == nullptr || table_pmax < pmax) return fail(-1, "factor tables must cover pmax%s");
  if (orth && (chain_off == nullptr || chain_q == nullptr)) return fail(-1, "orth needs chain tables%s");
  if (!periods || !powers || !status) return fail(-1, "output pointers are null%s");
  if (int rc = check_fold_mode(fold_mode)) return rc;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  const int hier = hier_applies(fold_mode, gamma ? PP_METRIC_GAMMA : PP_METRIC_NORM, trunc, orth) ? 1 : 0;
  const int f32 = (hier && !trunc && fold_mode == PP_FOLD_NOMINATE_F32) ? 1 : 0;
  const SmemPlan pl = make_plan(N, pmax, num, true, hier != 0, f32 != 0, true);
  const bool plain = !trunc && !orth;
  auto kernel = f32 ? mbest_kernel<true, true> : (plain ? mbest_kernel<false, true> : mbest_kernel<false, false>);
  if (int rc = prep_kernel(kernel, pl.bytes(), f)) return rc;
  const int grid = grid_for(f, pl.bytes(), B);
  size_t off = 0;
  double* slots = carve(workspace, workspace_bytes, off, (size_t)grid * num * pl.pv * 8);
  double* scr = orth ? carve(workspace, workspace_bytes, off, (size_t)grid * kWarps * 2 * pl.pv * 8) : nullptr;
  if (!slots || (orth && !scr)) return fail(-3, "workspace too small (see pp_workspace_bytes)%s");
  int* next_window = reinterpret_cast<int*>(carve(workspace, workspace_bytes, off, 256));
  if (!next_window) return fail(-3, "workspace too small (see pp_workspace_bytes)%s");
  if (int rc = check_cuda(cudaMemsetAsync(next_window, 0, sizeof(int), (cudaStream_t)stream), "cudaMemsetAsync")) return rc;
  uint2* tops = nullptr;
  int ntops = hier ? hier_top_count(pmin, pmax) : 0;
  if (ntops > 0) {
    tops = reinterpret_cast<uint2*>(carve(workspace, workspace_bytes, off, (size_t)ntops * sizeof(uint2)));
    if (!tops) return fail(-3, "workspace too small (see pp_workspace_bytes)%s");
    ntops = build_hier_jobs(N, pmin, pmax, hier_riders(fold_mode, trunc), tops, (cudaStream_t)stream);
  }
  Tables tb{chain_off, chain_q, fac_off, fac};
  kernel<<<grid, kThreads, pl.bytes(), (cudaStream_t)stream>>>(x, ldx, B, N, num, pmin, pmax, gamma, trunc, orth,
                                                                     hier, tb, periods, powers, bases, sweeps, status,
                                                                     slots, scr, tops, ntops, next_window,
                                                                     reinterpret_cast<unsigned long long*>(profile), f32,
                                                                     near_ties);
  return check_cuda(cudaGetLastError(), "mbest_kernel launch");
}

int pp_small_to_large(const double* x, int64_t ldx, int32_t B, int32_t N, double thresh, int32_t n_periods,
                      int32_t trunc, int32_t orth, const int32_t* chain_off, const int32_t* chain_q,
                      int32_t table_pmax, int32_t kmax, uint32_t* periods, double* powers, double* bases,
                      int32_t* count, int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (int rc = check_common(x, ldx, B, N)) return rc;
  if (!(thresh >= 0.0)) return fail(-1, "thresh must be >= 0%s");
  if (n_periods < 2 || n_periods > N) return fail(-1, "need 2 <= n_periods <= N%s");
  if (kmax < 1) return fail(-1, "kmax must be >= 1%s");
  if (orth && (chain_off == nullptr || chain_q == nullptr || table_pmax < n_periods)) return fail(-1, "orth needs tables covering n_periods%s");
  if (!periods || !powers || !count || !status) return fail(-1, "output pointers are null%s");
  if (B == 0) return 0;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  const SmemPlan pl = make_plan(N, n_periods, 0, true);
  if (int rc = prep_kernel(s2l_kernel, pl.bytes(), f)) return rc;
  const int grid = grid_for(f, pl.bytes(), B, kS2lCtasPerSm);
  size_t off = 0;
  double* scr = nullptr;
  if (orth) {
    scr = carve(workspace, workspace_bytes, off, (size_t)grid * kWarps * 2 * pl.pv * 8);
    if (!scr) return fail(-3, "workspace too small (see pp_workspace_bytes)%s");
  }
  Tables tb{chain_off, chain_q, nullptr, nullptr};
  int* next_window = carve_window_counter(workspace, workspace_bytes, off, (cudaStream_t)stream);
  s2l_kernel<<<grid, kThreads, pl.bytes(), (cudaStream_t)stream>>>(x, ldx, B, N, thresh, n_periods, trunc, orth, tb,
                                                                   kmax, periods, powers, bases, count, status, scr,
                                                                   next_window);
  return check_cuda(cudaGetLastError(), "s2l_kernel launch");
}

int pp_best_correlation(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t num, int32_t max_length,
                        double ratio, int32_t trunc, int32_t orth, int32_t fold_mode, const int32_t* chain_off,
                        const int32_t* chain_q, int32_t table_pmax, uint32_t* periods, double* powers, double* bases,
                        int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (int rc = check_common(x, ldx, B, N)) return rc;
  if (num < 1) return fail(-1, "num must be >= 1%s");
  if (max_length < 3 || max_length > N + 1) return fail(-1, "need 3 <= max_length <= N+1%s");
  if (orth && (chain_off == nullptr || chain_q == nullptr || table_pmax < max_length - 1)) return fail(-1, "orth needs tables covering max_length%s");
  if (!periods || !powers || !status) return fail(-1, "output pointers are null%s");
  if (int rc = check_fold_mode(fold_mode)) return rc;
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  // hierarchical ranking needs room for the per-CTA key arrays and the job table; without it: sequential folds
  size_t off = 0;
  int* next_window = carve_window_counter(workspace, workspace_bytes, off, (cudaStream_t)stream);
  int hier = fold_mode != PP_FOLD_DIRECT && max_length - 1 >= 4 ? 1 : 0;
  const size_t grid_max = (size_t)f.sm_count * kCtasPerSm;
  double* keys = nullptr;
  uint2* tops = nullptr;
  int ntops = 0;
  if (hier) {
    keys = carve(workspace, workspace_bytes, off, grid_max * (size_t)(max_length + 1) * 8);
    ntops = hier_top_count(2, max_length - 1);
    tops = reinterpret_cast<uint2*>(carve(workspace, workspace_bytes, off, (size_t)(ntops > 0 ? ntops : 1) * sizeof(uint2)));
    if (!keys || !tops || ntops <= 0) hier = 0;
  }
  const SmemPlan pl = make_plan(N, max_length, 0, true, hier != 0);
  if (int rc = prep_kernel(bcorr_kernel, pl.bytes(), f)) return rc;
  const int grid = grid_for(f, pl.bytes(), B);
  if (hier) ntops = build_hier_jobs(N, 2, max_length - 1, fold_mode != PP_FOLD_HIERARCHICAL_NO_RIDERS, tops, (cudaStream_t)stream);
  Tables tb{chain_off, chain_q, nullptr, nullptr};
  bcorr_kernel<<<grid, kThreads, pl.bytes(), (cudaStream_t)stream>>>(x, ldx, B, N, num, max_length, ratio, trunc, orth,
                                                                     tb, periods, powers, bases, status, next_window,
                                                                     hier, keys, tops, ntops);
  return check_cuda(cudaGetLastError(), "bcorr_kernel launch");
}

}  // extern "C"
