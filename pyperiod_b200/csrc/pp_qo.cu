// pyperiod_b200 -- QOPeriods on the B200: the quadratic-program residualisation of
// pyPeriod/QOPeriods.py:313-643, 743-852 as one persistent kernel.
//
// Per window (one CTA): up to `num` rounds of
//   gamma-norm sweep of the residual (QOPeriods.py:470-478; the sweep of pp_sweep.cuh)
//   -> dictionary layout: rows kept per period = sum of phi over newly seen divisors (:830-840)
//   -> normal equations  G w = W  with  G = A A^T (integer counts) and W = A x = fold sums of the
//      ORIGINAL data (:781-782), Cholesky in an L2-resident workspace, two triangular solves
//   -> reconstruction A^T w, residual = data - reconstruction (:517-522), stop test on
//      rms(reconstruction) (:391).
// The same solve stage serves RamanujanPeriods.find_periods_with_weights (RamanujanPeriods.py:106-112)
// through pp_qo_solve, and the rounds of a custom test_function through pp_qo_solve / pp_qo_solve_ramanujan.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pyperiod_b200.h"
#include "pp_common.cuh"
#include "pp_sweep.cuh"
#include "pp_chol.cuh"
#include "pp_cg.cuh"
#include "pp_host.cuh"

#include "pp_qo.cuh"

namespace pp {

// ------------------------------------------------------------------------------------------
// QOPeriods.find_periods, default branch (QOPeriods.py:313-596)
// ------------------------------------------------------------------------------------------
template <int BASIS>   // 0 natural (indicator rows, Cholesky), 1 Ramanujan sums (conjugate gradients)
__global__ void __launch_bounds__(kThreads, 2)
qo_find_kernel(QoBatch batch, int N, int num, double thresh, int pmin, int pmax, int trunc, int hier, int refine,
               const int32_t* __restrict__ phi, int rmax, QoOut out, unsigned char* __restrict__ ws, size_t ws_per_cta,
               const uint2* __restrict__ tops, int ntops, unsigned long long* __restrict__ prof,
               int* __restrict__ next_window) {
  unsigned char* smem = pp_smem;
  const QoPlan pl = make_qo_plan(N, pmax, num, rmax, hier != 0, BASIS == 1);
  unsigned char* ws_cta = ws + (size_t)blockIdx.x * ws_per_cta;
  QoCtx c = make_ctx(smem, pl, N, num, refine, phi, ws_cta);
  SweepShared* sweep = reinterpret_cast<SweepShared*>(smem + pl.off_sweep());
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + pl.off_bar());
  double* round_norms = reinterpret_cast<double*>(ws_cta + pl.ws_L() + pl.ws_save());
  double* x0 = const_cast<double*>(c.x0);
  const double sqrtN = sqrt((double)N);
  const int tid = threadIdx.x;
  long long timers[6] = {0, 0, 0, 0, 0, 0}, t_sweep = 0;
  c.t = timers;
  int done = 0;

  WindowLoader loader;
  loader.init(bar);
  sweep_shared_init(sweep);

  for (WindowQueue wq(next_window); wq.b < batch.count; wq.next()) {
    const int b = batch.window(wq.b);
    ++done;
    loader.load(x0, batch.x + (size_t)b * batch.ldx, N);
    // zero-signal early out (QOPeriods.py:394-406): sum |x| <= 1e-16
    double sa = 0.0;
    for (int n = tid; n < N; n += kThreads) {
      sa += fabs(x0[n]);
      c.xs[n] = x0[n];
    }
    for (int i = N + tid; i < pl.xs_len; i += kThreads) c.xs[i] = 0.0;  // the factorisation staged blocks here
    sa = warp_sum(sa);
    if ((tid & 31) == 0) c.red[tid >> 5] = sa;
    __syncthreads();
    double sum_abs = 0.0;
    for (int w = 0; w < kWarps; ++w) sum_abs += c.red[w];
    __syncthreads();
    const double e_data = cta_sum_sq(x0, N, c.red);
    // defaults: what the reference returns when nothing could be solved (empty lists, res = data)
    if (tid == 0) {
      c.misc[0] = 0;
      c.misc[1] = 0;
      c.misc[8] = 0;  // no Cholesky factor of this window in L yet
      c.misc[9] = 0;
      c.misc[11] = -1;  // no overflow-pool slot yet
    }
    __syncthreads();
    qo_commit(c, out, b, 0, round_norms);
    int status = PP_STATUS_OK;
    if (sum_abs <= 1e-16) {
      if (out.res)
        for (int n = tid; n < N; n += kThreads) out.res[(size_t)b * N + n] = 0.0;
      if (tid == 0) out.status[b] = PP_STATUS_ZERO_INPUT;
      __syncthreads();
      continue;
    }
    if (tid == 0) {
      SweepParams& sp = sweep->params;
      sp.N = N;
      sp.pmin = pmin;
      sp.pmax = pmax;
      sp.metric = PP_METRIC_GAMMA;
      sp.trunc = trunc;
      sp.orth = 0;  // QOPeriods.py:471-473 passes orthogonalize = False
      sp.chain_off = nullptr;
      sp.chain_q = nullptr;
      sp.warp_scr = nullptr;
      sp.pv = 0;
      sp.sqrtN = sqrtN;
      sp.e_res = 0.0;
      sp.data_norm = 1.0;
      sp.thresh = -1.0;
      sp.skip = nullptr;
      sp.nskip = 0;
      sp.metric_out = nullptr;
      sp.hier_scr = pl.hier_len ? reinterpret_cast<double*>(smem + pl.off_chol()) : nullptr;
      sp.hier_len = pl.hier_len;
      sp.rcp = sweep->rcp;
      sp.tops = tops;
      sp.ntops = ntops;
      sp.verify_keys = nullptr;
      sp.xf0_off = 0;
      sp.xf1_off = 0;
      sp.tie_keys = nullptr;
      sp.tie_nom = nullptr;
      sp.canon_v = nullptr;
      sp.canon_u = nullptr;
    }
    __syncthreads();
    int nfound = 0;
    int reported = 0;
    double e_recon = 0.0;
    const double rms_data = sqrt(e_data / (double)N);  // rms(), QOPeriods.py:78-79
    for (int i = 0; i < num; ++i) {
      if (i > 0) {
        // default test_function: rms(reconstruction) > rms(data) * thresh  (QOPeriods.py:391)
        const bool go = sqrt(e_recon / (double)N) > rms_data * thresh;
        if (!go) {
          // weights are re-solved with all periods (identical to what we hold) but the last period is
          // not reported (QOPeriods.py:560-594)
          reported = nfound > 0 ? nfound - 1 : 0;
          break;
        }
      }
      const long long t0 = clock64();
      const SweepResult top = cta_sweep<kSweepHier | kSweepNoMetricOut>(sweep);
      t_sweep += clock64() - t0;
      if (tid == 0) {
        round_norms[i] = top.val;
        if (top.p > 0) c.found[nfound] = top.p;
      }
      if (top.p > 0) ++nfound;
      __syncthreads();
      const int rc = BASIS == 1 ? cta_qo_solve_ram(c, nfound, &e_recon) : cta_qo_solve(c, nfound, &e_recon);
      if (rc != PP_STATUS_OK) {  // LinAlgError in the reference: keep the previous round's outputs (:552-559)
        status = rc;
        // the residual buffer may hold staged factor blocks: restore the padding the sweep relies on
        break;
      }
      // norms are indexed by round in the reference (norms[:len(found)]); rounds without a period only
      // happen once the residual is exactly zero, after which nothing changes
      if (!qo_commit(c, out, b, nfound, round_norms)) {  // overflow pool exhausted: the caller re-runs this window
        status = PP_STATUS_TOO_LARGE;
        if (tid == 0) out.n_weights[b] = c.misc[1];
        break;
      }
      reported = nfound;
      __syncthreads();
      // the factorisation used the residual buffer past N as staging space: the sweep reads zeros there
      for (int i2 = N + tid; i2 < pl.xs_len; i2 += kThreads) c.xs[i2] = 0.0;
      __syncthreads();
    }
    if (tid == 0) {
      out.n_periods[b] = status == PP_STATUS_OK ? reported : out.n_periods[b];
      out.status[b] = status;
    }
    __syncthreads();
  }
  if (prof != nullptr && tid == 0) {
    atomicAdd(prof + 0, (unsigned long long)t_sweep);
    atomicAdd(prof + 1, (unsigned long long)timers[0]);
    atomicAdd(prof + 2, (unsigned long long)timers[1]);
    atomicAdd(prof + 3, (unsigned long long)timers[2]);
    atomicAdd(prof + 5, (unsigned long long)timers[3]);
    atomicAdd(prof + 6, (unsigned long long)timers[4]);   // inside the factorisation: Gram counts
    atomicAdd(prof + 7, (unsigned long long)timers[5]);   // inside the factorisation: diagonal blocks (one warp)
    atomicAdd(prof + 4, (unsigned long long)done);
  }
}

// ------------------------------------------------------------------------------------------
// solve stage alone, for given periods (RamanujanPeriods.find_periods_with_weights :106-112) or for a
// caller-supplied dictionary layout (QOPeriodsWithGCDsExtracted.get_subspaces,
// QOPeriodsWithGCDsExtracted.py:98-143: that layout depends on CPython set order and is built on the host)
// ------------------------------------------------------------------------------------------
// explicit_rows == nullptr: entries[b, 0:n_entries[b]) are periods in the caller's order, the layout follows
// get_subspaces.  Otherwise entry k is the period entries[b, k] with its first explicit_rows[b, k] rows (0 = all).
// BASIS 1 (Ramanujan sums, conjugate gradients in the per-CTA workspace) takes periods only: explicit_rows == nullptr.
template <int BASIS>   // 0 natural (indicator rows, Cholesky), 1 Ramanujan sums (conjugate gradients)
__global__ void __launch_bounds__(kThreads, 2)
qo_solve_kernel(QoBatch batch, int N, int kmax, const int32_t* __restrict__ entries,
                const int32_t* __restrict__ explicit_rows, const int32_t* __restrict__ n_entries, int pmax, int refine,
                const int32_t* __restrict__ phi, int rmax, QoOut out, unsigned char* __restrict__ ws,
                size_t ws_per_cta, int* __restrict__ next_window, int x0_global) {
  unsigned char* smem = pp_smem;
  // x0_global: the window is read in place from global memory (L2) instead of being staged -- 32 KB less shared
  // memory, which is what lets dictionaries of up to N rows run two CTAs per SM (the factorisation of one window
  // is a latency-bound chain; the window itself is only read by the right-hand side and the residual)
  const QoPlan pl = make_qo_plan(N, pmax, kmax, rmax, false, BASIS == 1, x0_global != 0);
  QoCtx c = make_ctx(smem, pl, N, kmax, refine, phi, ws + (size_t)blockIdx.x * ws_per_cta);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + pl.off_bar());
  double* x0 = const_cast<double*>(c.x0);
  const int tid = threadIdx.x;
  long long timers[6] = {0, 0, 0, 0, 0, 0};
  c.t = timers;
  WindowLoader loader;
  loader.init(bar);
  for (WindowQueue wq(next_window); wq.b < batch.count; wq.next()) {
    const int b = batch.window(wq.b);
    if (x0_global) c.x0 = batch.x + (size_t)b * batch.ldx;
    else loader.load(x0, batch.x + (size_t)b * batch.ldx, N);
    const int nd = min(max(n_entries[b], 0), kmax);
    if (explicit_rows == nullptr) {
      for (int i = tid; i < nd; i += kThreads) c.found[i] = entries[(size_t)b * kmax + i];
      if (tid == 0) c.misc[8] = c.misc[9] = 0;  // one solve per window: nothing to extend
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
      // norms are the caller's (periodogram values); only layout, weights and residual are produced here
      if (out.dict_q != nullptr)
        for (int i = tid; i < kmax; i += kThreads) {
          out.dict_q[(size_t)b * kmax + i] = i < ndict ? c.dict_q[i] : 0;
          out.dict_keep[(size_t)b * kmax + i] = i < ndict ? c.dict_keep[i] : 0;
        }
      double* w = out.weights_of(b);
      for (int i = tid; i < R; i += kThreads) w[i] = c.wv[i];
      if (out.res)
        for (int n = tid; n < N; n += kThreads) out.res[(size_t)b * N + n] = c.xs[n];
    } else if (out.res) {
      // not solved (singular / too large): nothing was explained, the residual is the data (the reference raises here)
      for (int n = tid; n < N; n += kThreads) out.res[(size_t)b * N + n] = c.x0[n];
    }
    if (tid == 0) {
      if (out.n_dict != nullptr) out.n_dict[b] = rc == PP_STATUS_OK ? ndict : 0;
      // a window that did not fit reports the rows it needs, so the caller can size a second launch
      out.n_weights[b] = rc == PP_STATUS_OK ? R : (rc == PP_STATUS_TOO_LARGE ? R : 0);
      out.status[b] = rc;
    }
    __syncthreads();
  }
}

// rows of the dictionary get_subspaces builds for the given periods (QOPeriods.py:830-840): rows[b] = sum of the
// rows kept per period.  Lets the caller size the factor storage before pp_qo_solve.
__global__ void __launch_bounds__(kThreads)
qo_rows_kernel(int B, int kmax, const int32_t* __restrict__ periods, const int32_t* __restrict__ nper, int pmax,
               const int32_t* __restrict__ phi, int32_t* __restrict__ rows_out) {
  extern __shared__ uint32_t qr_seen[];   // bitmap of divisors, then kmax periods already in the dictionary
  const int words = (pmax + 32) / 32;
  int* seen_q = reinterpret_cast<int*>(qr_seen + words);
  __shared__ int s_fresh, s_total, s_nd;
  const int tid = threadIdx.x;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    for (int i = tid; i < words; i += kThreads) qr_seen[i] = 0u;
    if (tid == 0) s_total = s_nd = 0;
    __syncthreads();
    const int nf = min(max(nper[b], 0), kmax);
    for (int f = 0; f < nf; ++f) {
      const int q = periods[(size_t)b * kmax + f];
      if (tid == 0) s_fresh = 0;
      __syncthreads();
      int fresh = 0;
      for (int d = 1 + tid; d <= q; d += kThreads)
        if (q % d == 0 && !((qr_seen[d >> 5] >> (d & 31)) & 1u)) {
          fresh += phi[d];
          atomicOr(&qr_seen[d >> 5], 1u << (d & 31));
        }
      if (fresh) atomicAdd(&s_fresh, fresh);
      __syncthreads();
      if (tid == 0) {
        // a repeated period keeps 0 new rows and then contributes all q of them (QOPeriods.py:972); its earlier
        // contribution is replaced
        int slot = -1;
        for (int k = 0; k < s_nd; ++k)
          if (seen_q[2 * k] == q) slot = k;
        const int rows = s_fresh ? s_fresh : q;
        if (slot < 0) {
          slot = s_nd++;
          seen_q[2 * slot] = q;
          seen_q[2 * slot + 1] = 0;
        }
        s_total += rows - seen_q[2 * slot + 1];
        seen_q[2 * slot + 1] = rows;
      }
      __syncthreads();
    }
    if (tid == 0) rows_out[b] = s_total;
    __syncthreads();
  }
}

}  // namespace pp

using namespace pp;

extern "C" {

size_t pp_qo_workspace_bytes(int32_t N, int32_t pmax, int32_t num, int32_t rmax, int32_t ctas, int32_t basis) {
  DeviceFacts f;
  if (device_facts(f)) return 0;
  const QoPlan pl = make_qo_plan(N, pmax, num, rmax, true, basis == PP_BASIS_RAMANUJAN);
  // the solve kernel may keep the window in global memory to fit a second CTA per SM: size for the full grid
  size_t grid = (size_t)kQoCtasPerSm * (size_t)f.sm_count;
  if (basis == PP_BASIS_RAMANUJAN) grid = (size_t)grid_for(f, pl.bytes(), 0, kQoCtasPerSm);
  if (ctas > 0 && (size_t)ctas < grid) grid = (size_t)ctas;
  return 8192 + (size_t)(pmax + 2) * sizeof(uint2) + grid * pl.ws_per_cta();
}

static int qo_check(const void* x, int64_t ldx, int B, int N, int num, int pmax, int rmax, const void* phi,
                    int table_pmax) {
  if (x == nullptr || B < 0 || N < 2 || ldx < 1) return fail(-1, "bad window arguments%s");
  if (num < 1 || num > 256) return fail(-1, "need 1 <= num <= 256%s");
  if (pmax < 1 || pmax > N) return fail(-1, "need 1 <= pmax <= N%s");
  if (pmax > 32767 || N > 32767) return fail(-1, "periods and windows above 32767 samples are not supported%s");
  if (rmax < 2) return fail(-1, "rmax must be >= 2%s");
  if (table_pmax >= 0 && (phi == nullptr || table_pmax < pmax)) return fail(-1, "phi table must cover pmax%s");
  return 0;
}

// persistent grid of a QO launch: limited by shared memory, the batch, and the factor storage the workspace holds
static int qo_grid(const DeviceFacts& f, const QoPlan& pl, int count, size_t avail_bytes) {
  int grid = grid_for(f, pl.bytes(), count, kQoCtasPerSm);
  const size_t fit = avail_bytes / pl.ws_per_cta();
  if ((size_t)grid > fit) grid = (int)fit;
  return grid;
}

int pp_qo_find_periods(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t num, double thresh, int32_t pmin,
                       int32_t pmax, int32_t trunc, int32_t fold_mode, int32_t refine, int32_t basis,
                       const int32_t* phi, int32_t table_pmax, int32_t rmax, const int32_t* order, int32_t n_order,
                       uint32_t* periods,
                       double* norms, int32_t* n_periods, int32_t* dict_q, int32_t* dict_keep, int32_t* n_dict,
                       int32_t* n_weights, double* weights, int64_t ldw, double* res, int32_t* status,
                       double* weights_pool, int32_t pool_slots, int32_t* pool_slot, void* workspace,
                       size_t workspace_bytes, void* profile, void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  const int count = order ? n_order : B;
  if (count == 0) return 0;
  if (int rc = qo_check(x, ldx, B, N, num, pmax, rmax, phi, table_pmax)) return rc;
  if (num > 64) return fail(-1, "need num <= 64%s");
  if (pmin < 1 || pmin > pmax) return fail(-1, "need 1 <= pmin <= pmax%s");
  if (refine < 0 || refine > 4) return fail(-1, "refine must be in [0, 4]%s");
  if (!periods || !norms || !n_periods || !dict_q || !dict_keep || !n_dict || !n_weights || !weights || !status)
    return fail(-1, "output pointers are null%s");
  if (count < 0 || count > B) return fail(-1, "bad order list%s");
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  if (int rc = check_fold_mode(fold_mode)) return rc;
  const int hier = (fold_mode != PP_FOLD_DIRECT && !trunc) ? 1 : 0;
  if (basis != PP_BASIS_NATURAL && basis != PP_BASIS_RAMANUJAN) return fail(-1, "unknown basis%s");
  const bool ram = basis == PP_BASIS_RAMANUJAN;
  const QoPlan pl = make_qo_plan(N, pmax, num, rmax, hier != 0, ram);
  const bool pooled = weights_pool != nullptr && !ram;
  if (pooled) {
    if (pool_slot == nullptr || pool_slots < 1 || ldw < 32) return fail(-1, "bad overflow pool arguments%s");
  } else if (ldw < pl.rmax) {
    return fail(-1, "ldw must be >= rmax rounded up to a multiple of 32 (or pass a weights pool)%s");
  }
  if (int rc = ram ? prep_kernel(qo_find_kernel<1>, pl.bytes(), f) : prep_kernel(qo_find_kernel<0>, pl.bytes(), f))
    return rc;
  size_t off = 0;
  int* next_window = carve_window_counter(workspace, workspace_bytes, off, (cudaStream_t)stream);
  int* pool_counter = pooled ? carve_window_counter(workspace, workspace_bytes, off, (cudaStream_t)stream) : nullptr;
  if (pooled && pool_counter == nullptr) return fail(-3, "workspace too small (see pp_qo_workspace_bytes)%s");
  uint2* tops = nullptr;
  int ntops = hier ? hier_top_count(pmin, pmax) : 0;
  if (ntops > 0) {
    tops = reinterpret_cast<uint2*>(carve(workspace, workspace_bytes, off, (size_t)ntops * sizeof(uint2)));
    if (!tops) return fail(-3, "workspace too small (see pp_qo_workspace_bytes)%s");
    ntops = build_hier_jobs(N, pmin, pmax, fold_mode != PP_FOLD_HIERARCHICAL_NO_RIDERS, tops, (cudaStream_t)stream);
  }
  off = (off + 255) & ~(size_t)255;
  if (workspace == nullptr || next_window == nullptr || off >= workspace_bytes)
    return fail(-3, "workspace too small (see pp_qo_workspace_bytes)%s");
  const int grid = qo_grid(f, pl, count, workspace_bytes - off);
  if (grid < 1) return fail(-3, "workspace too small for one factor (see pp_qo_workspace_bytes)%s");
  QoOut o{periods, norms, n_periods, dict_q, dict_keep, n_dict, n_weights, weights, nullptr, ldw, res, status};
  if (pooled) {
    o.pool = weights_pool;
    o.pool_slots = pool_slots;
    o.pool_stride = pl.rmax;
    o.pool_counter = pool_counter;
    o.pool_slot = pool_slot;
  }
  QoBatch batch{x, ldx, count, order};
  if (ram)
    qo_find_kernel<1><<<grid, kThreads, pl.bytes(), (cudaStream_t)stream>>>(
        batch, N, num, thresh, pmin, pmax, trunc, hier, refine, phi, pl.rmax, o,
        reinterpret_cast<unsigned char*>(workspace) + off, pl.ws_per_cta(), tops, ntops,
        reinterpret_cast<unsigned long long*>(profile), next_window);
  else
    qo_find_kernel<0><<<grid, kThreads, pl.bytes(), (cudaStream_t)stream>>>(
        batch, N, num, thresh, pmin, pmax, trunc, hier, refine, phi, pl.rmax, o,
        reinterpret_cast<unsigned char*>(workspace) + off, pl.ws_per_cta(), tops, ntops,
        reinterpret_cast<unsigned long long*>(profile), next_window);
  return check_cuda(cudaGetLastError(), "qo_find_kernel launch");
}

// plan of qo_solve_kernel: the window is kept in global memory when that is what makes room for a second CTA per SM
static QoPlan qo_solve_plan(const DeviceFacts& f, int N, int pmax, int kmax, int rmax, int& x0_global, bool ram = false) {
  QoPlan pl = make_qo_plan(N, pmax, kmax, rmax, false, ram);
  x0_global = 0;
  if (grid_for(f, pl.bytes(), 0, kQoCtasPerSm) < kQoCtasPerSm * f.sm_count) {
    const QoPlan alt = make_qo_plan(N, pmax, kmax, rmax, false, ram, true);
    if (grid_for(f, alt.bytes(), 0, kQoCtasPerSm) > grid_for(f, pl.bytes(), 0, kQoCtasPerSm)) {
      pl = alt;
      x0_global = 1;
    }
  }
  return pl;
}

static int qo_solve_launch(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t* entries,
                           const int32_t* explicit_rows, const int32_t* n_entries, int32_t pmax, int32_t refine,
                           const int32_t* phi, int32_t rmax, const int32_t* order, int32_t n_order, QoOut o,
                           void* workspace, size_t workspace_bytes, void* stream, bool ram = false) {
  const int count = order ? n_order : B;
  if (count == 0) return 0;
  if (count < 0 || count > B) return fail(-1, "bad order list%s");
  if (refine < 0 || refine > 4) return fail(-1, "refine must be in [0, 4]%s");
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  int x0_global = 0;
  const QoPlan pl = qo_solve_plan(f, N, pmax, kmax, rmax, x0_global, ram);
  if (o.weights_off == nullptr && o.ldw < pl.rmax)
    return fail(-1, "ldw must be >= rmax rounded up to a multiple of 32 (or pass weights_off)%s");
  if (int rc = ram ? prep_kernel(qo_solve_kernel<1>, pl.bytes(), f) : prep_kernel(qo_solve_kernel<0>, pl.bytes(), f))
    return rc;
  size_t off = 0;
  int* next_window = carve_window_counter(workspace, workspace_bytes, off, (cudaStream_t)stream);
  off = (off + 255) & ~(size_t)255;
  if (workspace == nullptr || next_window == nullptr || off >= workspace_bytes)
    return fail(-3, "workspace too small (see pp_qo_workspace_bytes)%s");
  const int grid = qo_grid(f, pl, count, workspace_bytes - off);
  if (grid < 1) return fail(-3, "workspace too small for one factor (see pp_qo_workspace_bytes)%s");
  QoBatch batch{x, ldx, count, order};
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace) + off;
  if (ram)
    qo_solve_kernel<1><<<grid, kThreads, pl.bytes(), (cudaStream_t)stream>>>(
        batch, N, kmax, entries, nullptr, n_entries, pmax, refine, phi, pl.rmax, o, ws, pl.ws_per_cta(), next_window,
        x0_global);
  else
    qo_solve_kernel<0><<<grid, kThreads, pl.bytes(), (cudaStream_t)stream>>>(
        batch, N, kmax, entries, explicit_rows, n_entries, pmax, refine, phi, pl.rmax, o, ws, pl.ws_per_cta(),
        next_window, x0_global);
  return check_cuda(cudaGetLastError(), "qo_solve_kernel launch");
}

int pp_qo_solve(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t* periods,
                const int32_t* nper, int32_t pmax, int32_t refine, const int32_t* phi, int32_t table_pmax,
                int32_t rmax, const int32_t* order, int32_t n_order, int32_t* dict_q, int32_t* dict_keep,
                int32_t* n_dict, int32_t* n_weights, double* weights, int64_t ldw, const int64_t* weights_off,
                double* res, int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (int rc = qo_check(x, ldx, B, N, kmax, pmax, rmax, phi, table_pmax)) return rc;
  if (!periods || !nper || !dict_q || !dict_keep || !n_dict || !n_weights || !weights || !status)
    return fail(-1, "pointers are null%s");
  QoOut o{nullptr, nullptr, nullptr, dict_q, dict_keep, n_dict, n_weights, weights, weights_off, ldw, res, status};
  return qo_solve_launch(x, ldx, B, N, kmax, periods, nullptr, nper, pmax, refine, phi, rmax, order, n_order, o,
                         workspace, workspace_bytes, stream);
}

int pp_qo_solve_ramanujan(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t* periods,
                          const int32_t* nper, int32_t pmax, int32_t refine, const int32_t* phi, int32_t table_pmax,
                          int32_t rmax, const int32_t* order, int32_t n_order, int32_t* dict_q, int32_t* dict_keep,
                          int32_t* n_dict, int32_t* n_weights, double* weights, int64_t ldw, const int64_t* weights_off,
                          double* res, int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (int rc = qo_check(x, ldx, B, N, kmax, pmax, rmax, phi, table_pmax)) return rc;
  if (!periods || !nper || !dict_q || !dict_keep || !n_dict || !n_weights || !weights || !status)
    return fail(-1, "pointers are null%s");
  QoOut o{nullptr, nullptr, nullptr, dict_q, dict_keep, n_dict, n_weights, weights, weights_off, ldw, res, status};
  return qo_solve_launch(x, ldx, B, N, kmax, periods, nullptr, nper, pmax, refine, phi, rmax, order, n_order, o,
                         workspace, workspace_bytes, stream, true);
}

int pp_qo_solve_rows(const double* x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t* dict_q,
                     const int32_t* dict_rows, const int32_t* n_dict, int32_t pmax, int32_t refine, int32_t rmax,
                     int32_t* n_weights, double* weights, int64_t ldw, double* res, int32_t* status, void* workspace,
                     size_t workspace_bytes, void* stream) {
  if (B == 0) return 0;  // empty batch: nothing to validate or launch
  if (int rc = qo_check(x, ldx, B, N, kmax, pmax, rmax, nullptr, -1)) return rc;
  if (!dict_q || !dict_rows || !n_dict || !n_weights || !weights || !status) return fail(-1, "pointers are null%s");
  QoOut o{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, n_weights, weights, nullptr, ldw, res, status};
  return qo_solve_launch(x, ldx, B, N, kmax, dict_q, dict_rows, n_dict, pmax, refine, nullptr, rmax, nullptr, 0, o,
                         workspace, workspace_bytes, stream);
}

int pp_qo_fits_on_chip(int32_t kind, int32_t N, int32_t pmax, int32_t num, int32_t rmax, int32_t basis,
                       int32_t fold_mode, int32_t smem_bytes) {
  if (N < 2 || pmax < 1 || num < 1 || rmax < 2 || smem_bytes < 0) return fail(-1, "bad arguments%s");
  if (basis != PP_BASIS_NATURAL && basis != PP_BASIS_RAMANUJAN) return fail(-1, "unknown basis%s");
  if (check_fold_mode(fold_mode)) return -1;
  const size_t smem = (size_t)smem_bytes;
  if (kind == PP_QO_KIND_MURESAN) return muresan_smem_bytes(N, pmax) <= smem ? 1 : 0;
  if (kind != PP_QO_KIND_FIND && kind != PP_QO_KIND_SOLVE && kind != PP_QO_KIND_SOLVE_RAMANUJAN)
    return fail(-1, "unknown kind%s");
  // the solve kinds name their basis: a basis argument that contradicts the kind is rejected
  if (kind == PP_QO_KIND_SOLVE && basis != PP_BASIS_NATURAL)
    return fail(-1, "PP_QO_KIND_SOLVE is the natural-basis solve stage (see PP_QO_KIND_SOLVE_RAMANUJAN)%s");
  if (kind == PP_QO_KIND_SOLVE_RAMANUJAN && basis != PP_BASIS_RAMANUJAN)
    return fail(-1, "PP_QO_KIND_SOLVE_RAMANUJAN needs basis PP_BASIS_RAMANUJAN%s");
  // qo_check: the hierarchical fold's job descriptors hold N / g and N mod g in 16 bits
  if (N > 32767 || pmax > 32767) return 0;
  if (kind == PP_QO_KIND_FIND) {
    // the find kernel folds directly under trunc: callers pass PP_FOLD_DIRECT for a trunc call
    const bool hier = fold_mode != PP_FOLD_DIRECT;
    return make_qo_plan(N, pmax, num, rmax, hier, basis == PP_BASIS_RAMANUJAN).bytes() <= smem ? 1 : 0;
  }
  DeviceFacts f;   // the choice of qo_solve_plan depends on the shared memory per SM only, not on the SM count
  f.sm_count = 1;
  f.smem_optin = smem_bytes;
  int x0_global = 0;
  return qo_solve_plan(f, N, pmax, num, rmax, x0_global, kind == PP_QO_KIND_SOLVE_RAMANUJAN).bytes() <= smem ? 1 : 0;
}

int pp_qo_dictionary_rows(int32_t B, int32_t kmax, const int32_t* periods, const int32_t* nper, int32_t pmax,
                          const int32_t* phi, int32_t table_pmax, int32_t* rows, void* stream) {
  if (B == 0) return 0;
  if (B < 0 || kmax < 1 || !periods || !nper || !rows) return fail(-1, "bad arguments%s");
  if (pmax < 1 || phi == nullptr || table_pmax < pmax) return fail(-1, "phi table must cover pmax%s");
  DeviceFacts f;
  if (int rc = device_facts(f)) return rc;
  const size_t smem = (size_t)((pmax + 32) / 32) * 4 + (size_t)kmax * 8;
  if (smem > 48 * 1024)
    if (int rc = prep_kernel(qo_rows_kernel, smem, f)) return rc;
  int grid = f.sm_count * 8;
  if (grid > B) grid = B;
  qo_rows_kernel<<<grid, kThreads, smem, (cudaStream_t)stream>>>(B, kmax, periods, nper, pmax, phi, rows);
  return check_cuda(cudaGetLastError(), "qo_rows_kernel launch");
}

}  // extern "C"
