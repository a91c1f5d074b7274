/*
 * pyperiod_b200 -- C ABI of the B200-native periodicity-projection hot path.
 *
 * The reference (woolgathering/pyPeriod) is pure Python; it has no FFI.  The drop-in
 * boundary is its Python class API, and this header is what the Python layer
 * (pyperiod_b200/*.py, ctypes) binds underneath it.  Each entry point names the
 * reference interface it replaces (file:line relative to the reference root).
 *
 * Conventions
 *  - extern "C", plain pointers and sizes; no C++ or torch types cross the edge.
 *  - Every data pointer is a DEVICE pointer unless the name ends in `_host`.
 *  - x is a batch of B windows of N float64 samples; window b starts at x + b*ldx
 *    (ldx in ELEMENTS; ldx < N is allowed and means overlapping windows cut from one
 *    stream, e.g. ldx = hop = 512 for config 3).
 *  - `stream` is a cudaStream_t passed as void*; calls only enqueue work (no sync)
 *    unless documented.  The library allocates nothing the caller must free:
 *    workspaces are caller-owned, sized by pp_workspace_bytes().
 *  - Return value: 0 on success, <0 on argument / CUDA error (text via
 *    pp_last_error()).  Data-dependent outcomes (no period found, singular Gram, kmax
 *    overflow) go to the per-window int32 status[B] output, never to the return code.
 *  - Integer side tables (pp_tables_*) are built on the host by evaluating the
 *    reference's own divisor-set expression, because CPython set iteration order
 *    decides the orthogonalisation order and M-best step 2 (SURVEY.md 8a row 3).
 */
#ifndef PYPERIOD_B200_H
#define PYPERIOD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PP_ABI_VERSION 11

/* sweep metrics */
#define PP_METRIC_NORM 0   /* ||proj_p|| / sqrt(N)                 Periods.py:221-241, 507-508 */
#define PP_METRIC_GAMMA 1  /* ... / sqrt(p)                        Periods.py:239, 509-510      */
#define PP_METRIC_MAXABS 2 /* max_s |sum x[s::p]|                  Periods.py:327-331           */
#define PP_METRIC_IMPOSED 3 /* (||r|| - ||r - proj_p r||)/||x||    Periods.py:278-280           */

/* per-window status codes */
#define PP_STATUS_OK 0
#define PP_STATUS_NO_PERIOD 1   /* sweep found no positive metric (reference raises TypeError) */
#define PP_STATUS_OVERFLOW 2    /* more accepted periods than kmax (small_to_large)            */
#define PP_STATUS_SINGULAR 3    /* Gram matrix not positive definite (reference: LinAlgError)  */
#define PP_STATUS_GUARD 4       /* iteration guard tripped                                     */
#define PP_STATUS_TOO_LARGE 5   /* dictionary has more rows than rmax                          */
#define PP_STATUS_ZERO_INPUT 6  /* sum |x| <= 1e-16: the reference returns a canned result     */

/* workspace selector for pp_workspace_bytes */
#define PP_ALGO_SWEEP 0
#define PP_ALGO_MBEST 1
#define PP_ALGO_S2L 2
#define PP_ALGO_BCORR 3
#define PP_ALGO_QO 4
#define PP_ALGO_RAMANUJAN 5
#define PP_ALGO_PROJECT 6
#define PP_ALGO_BFREQ 7

int pp_abi_version(void);
const char *pp_last_error(void);

/* How ranking sweeps (NORM / GAMMA, no trunc, no orth) obtain the residue sums:
 *   PP_FOLD_HIERARCHICAL (default): only periods in (pmax/2, pmax] are folded from the window;
 *       S_p for smaller p follows from S_2p[r] + S_2p[r+p].  Half the shared-memory traffic;
 *       energies differ from the sequential fold by rounding only (a few ulp).
 *       Tops that are 3/2 or 3/4 of an even top q = g 2^L (g odd, L in {1, 2}) ride on q's pass
 *       (3 * 2^L accumulator sets at base g), which saves about a fifth of the passes.
 *   PP_FOLD_DIRECT: every candidate period is folded sequentially from the window.
 *   PP_FOLD_HIERARCHICAL_NO_RIDERS: hierarchical, one pass per top (for comparisons).
 *   PP_FOLD_NOMINATE_F32: M-best ranks with the hierarchical sweep in float (half the shared-memory
 *       traffic), then folds every candidate whose error bound reaches the best one sequentially in fp64:
 *       the selected periods and norms are those of the exact fold.
 * Outputs that must be bit-exact (project(), the bases, MAXABS metrics) never use the
 * hierarchical sums.  The mode is an argument of every call that sweeps (`fold_mode`): the library keeps no
 * process-wide state, so calls on different streams / threads do not influence each other. */
#define PP_FOLD_HIERARCHICAL 0
#define PP_FOLD_DIRECT 1
#define PP_FOLD_HIERARCHICAL_NO_RIDERS 2
#define PP_FOLD_NOMINATE_F32 3
/* Passes over a window of N samples one ranking sweep of [pmin, pmax] executes under `fold_mode`
 * (pmax - pmin + 1 for PP_FOLD_DIRECT; tops minus riders for PP_FOLD_HIERARCHICAL). */
int pp_sweep_passes(int32_t N, int32_t pmin, int32_t pmax, int32_t fold_mode);

/* `profile` arguments (development aid, nullable): a device buffer of 8 uint64 to which the call adds
 * SM-cycle counts.  pp_mbest: [0] sweeps, [1] exact winner projections, [2] bookkeeping + residual update,
 * [3] step 2 + outputs, [4] windows.  pp_qo_find_periods: [0] sweeps, [1] dictionary layout, [2] right-hand
 * side + pair tables, [3] Cholesky factorisation (tensor cores), [5] triangular solves + reconstruction (+
 * refinement), [4] windows. */

/* Device facts the host uses for grid sizing / roofline arithmetic (current device). */
int pp_device_info(int32_t *sm_count, int32_t *smem_optin_bytes, int32_t *cc_major, int32_t *cc_minor,
                   int32_t *clock_khz);

/* Number of persistent CTAs the library launches for this shape (grid size), and the
 * caller-owned workspace it needs.  `orth` matters because orthogonalised sweeps use a
 * per-warp global scratch. */
int pp_grid_size(int32_t algo, int32_t N, int32_t pmax, int32_t orth);
size_t pp_workspace_bytes(int32_t algo, int32_t N, int32_t pmax, int32_t num, int32_t orth);

/* Integer side tables (device arrays, indexed by period p in [0, table_pmax]):
 *   chain_off[p] .. chain_off[p+1] : cofactors p//f, f prime divisor of p, reference set order
 *                                    (Periods.py:208-214)
 *   fac_off[p] .. fac_off[p+1]     : non-trivial divisors of p, reference set order
 *                                    (Periods.py:548-549)
 * Passed as five arguments wherever a call may orthogonalise or run M-best step 2. */

/* ---- Periods.project (Periods.py:142-219) -------------------------------------------
 * out[b, 0:out_len] = project(x[b], p, trunc, orth)[0:out_len]; out_len = N, or p for
 * return_single_period.  chain_q_host[0:chain_len] = cofactors for this p (empty = no
 * orthogonalisation).  Bit-exact with the reference's numpy arithmetic. */
int pp_project(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t p, int32_t trunc,
               const int32_t *chain_q_host, int32_t chain_len, double *out, int64_t ldo, int32_t out_len,
               void *stream);

/* ---- Periods.periodic_norm (Periods.py:221-241) -------------------------------------
 * out[b] = ||x_b||_2 / sqrt(N), additionally / sqrt(p) when p > 0 (the "gamma" norm). */
int pp_periodic_norm(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t p, double *out, void *stream);

/* ---- one sweep over p in [pmin, pmax] (inner loops of Periods.py:501-515, 324-331,
 *      QOPeriods.py:470-478) ------------------------------------------------------------
 * metric_out (nullable): [B, pmax+1] row-major, entries below pmin untouched.
 * best_p / best_val: strict-'>' argmax from 0 in ascending p (lowest p wins ties); best_p = 0
 * when no metric is positive.  PP_METRIC_IMPOSED is evaluated against the window itself
 * as both residual and data (thresholding is done by pp_small_to_large). */
int pp_sweep(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t pmin, int32_t pmax, int32_t metric,
             int32_t trunc, int32_t orth, int32_t fold_mode, const int32_t *chain_off, const int32_t *chain_q,
             int32_t table_pmax, double *metric_out, int32_t *best_p, double *best_val, void *workspace,
             size_t workspace_bytes, void *stream);

/* ---- Periods.m_best / m_best_gamma (Periods.py:408-601) -------------------------------
 * periods[B,num] u32, powers[B,num] f64, bases[B,num,N] f64 (nullable: bases stay on chip /
 * in the workspace), sweeps[B] = step-1 sweeps executed (nullable), status[B].
 * near_ties[B] (nullable) = number of step-1 sweeps in which more than one candidate lay within the rounding
 * bound of the best ranking value; those sweeps are decided by the exact re-ranking (sequential fold, IEEE
 * mean, fixed-order sum of squares of the tiled base, strict '>' in ascending p -- Periods.py:507-515), so the
 * selected period does not depend on the fold mode.  On inputs with a noise floor it is 0. */
int pp_mbest(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t num, int32_t pmin, int32_t pmax,
             int32_t gamma, int32_t trunc, int32_t orth, int32_t fold_mode, const int32_t *chain_off,
             const int32_t *chain_q, const int32_t *fac_off, const int32_t *fac, int32_t table_pmax,
             uint32_t *periods, double *powers, double *bases, int32_t *sweeps, int32_t *near_ties,
             int32_t *status, void *workspace, size_t workspace_bytes, void *profile, void *stream);

/* ---- Periods.small_to_large (Periods.py:246-287) --------------------------------------
 * p runs 2..n_periods; periods[B,kmax] u32, powers[B,kmax], bases[B,kmax,N] (nullable),
 * count[B] = number accepted (may exceed kmax: then status = PP_STATUS_OVERFLOW and only
 * the first kmax are stored). */
int pp_small_to_large(const double *x, int64_t ldx, int32_t B, int32_t N, double thresh, int32_t n_periods,
                      int32_t trunc, int32_t orth, const int32_t *chain_off, const int32_t *chain_q,
                      int32_t table_pmax, int32_t kmax, uint32_t *periods, double *powers, double *bases,
                      int32_t *count, int32_t *status, void *workspace, size_t workspace_bytes, void *stream);

/* ---- Periods.best_correlation (Periods.py:289-349) ------------------------------------
 * candidates p in [2, max_length) (max_length excluded, :324); rejected rounds leave
 * periods/powers/bases rows at zero.  With a workspace of pp_workspace_bytes(PP_ALGO_BCORR, N,
 * max_length, num, orth) bytes the sweep nominates hierarchically and verifies with sequential folds
 * (bit-identical results, about twice as fast); with workspace == NULL every candidate is folded
 * sequentially. */
int pp_best_correlation(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t num, int32_t max_length,
                        double ratio, int32_t trunc, int32_t orth, int32_t fold_mode, const int32_t *chain_off,
                        const int32_t *chain_q, int32_t table_pmax, uint32_t *periods, double *powers,
                        double *bases, int32_t *status, void *workspace, size_t workspace_bytes, void *stream);

/* ---- Periods.best_frequency (Periods.py:351-398), one round for a batch ---------------------------------
 * mags[B, F]: magnitude spectrum of the current residual (|rfft(work, win_size)|, F = win_size / 2 + 1; the FFT
 * itself is the FFT library's).  Per window: bin = first arg-max of mags (np.argmax), p = round-half-even(2 *
 * win_size / bin) (:383-386), base = project(work, p, trunc, orth) bit-exactly, periods[b, round] = p,
 * norms[b, round] = ||base|| / sqrt(N), bases[b, round, :] = base (nullable), work[b] -= base in place.  Every
 * window has its own period in the same launch.  status[b] must be PP_STATUS_OK on entry of round 0; a window
 * whose peak is the DC bin gets PP_STATUS_NO_PERIOD (the reference raises OverflowError on int(round(inf))) and
 * is skipped by later rounds.  p > N is the reference's one-row padding case (:172-176). */
int pp_best_frequency_round(double *work, int32_t B, int32_t N, const double *mags, int32_t F, int32_t win_size,
                            int32_t trunc, int32_t orth, const int32_t *chain_off, const int32_t *chain_q,
                            int32_t table_pmax, uint32_t *periods, double *norms, double *bases, int32_t round,
                            int32_t num, int32_t *status, void *stream);

/* ---- the global-memory ("long") path of the Periods family -------------------------------------------------
 * The on-chip entry points above stage the whole window, the single-period vectors and the sweep scratch of one
 * window in one CTA's shared memory and return -2 when that plan does not fit.  pp_fits_on_chip answers, without
 * touching a device, whether the on-chip plan of a call fits `smem_bytes` (the device's opt-in shared memory per
 * block): 1 = fits, 0 = does not, < 0 = bad arguments.  algo: PP_ALGO_PROJECT (pmax = p), PP_ALGO_SWEEP,
 * PP_ALGO_MBEST (metric NORM or GAMMA), PP_ALGO_S2L (pmax = n_periods), PP_ALGO_BCORR (pmax = max_length) or
 * PP_ALGO_BFREQ (pmax unused); metric / trunc / orth / fold_mode are the call's own (they decide which sweep
 * scratch the plan holds).
 *
 * pp_long_* take the arguments of the on-chip entry point of the same name and return the same results for any
 * window length: residuals are copied to the workspace (the input is never written), every sweep is spread over the
 * whole GPU as one work unit per (window, candidate period), and each window's selection step runs in one CTA.  The
 * host drives the rounds on `stream` and reads a 4-byte active-window count once per round, so these calls return
 * after their work is done except pp_long_project and pp_long_best_frequency_round, which only enqueue.  Ranking
 * sweeps fold directly (sequential fp64 sums, the fold_mode of the on-chip call has no counterpart), so M-best in
 * every fold mode and dtype selects the periods and powers of the fp64 direct fold.  Workspace:
 * pp_long_workspace_bytes(algo, B, N, pmax, num, orth), with pmax as for pp_fits_on_chip (N for PP_ALGO_BFREQ). */
int pp_fits_on_chip(int32_t algo, int32_t N, int32_t pmax, int32_t num, int32_t metric, int32_t trunc, int32_t orth,
                    int32_t fold_mode, int32_t smem_bytes);
size_t pp_long_workspace_bytes(int32_t algo, int32_t B, int32_t N, int32_t pmax, int32_t num, int32_t orth);
int pp_long_project(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t p, int32_t trunc,
                    const int32_t *chain_q_host, int32_t chain_len, double *out, int64_t ldo, int32_t out_len,
                    void *workspace, size_t workspace_bytes, void *stream);
int pp_long_sweep(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t pmin, int32_t pmax, int32_t metric,
                  int32_t trunc, int32_t orth, const int32_t *chain_off, const int32_t *chain_q, int32_t table_pmax,
                  double *metric_out, int32_t *best_p, double *best_val, void *workspace, size_t workspace_bytes,
                  void *stream);
int pp_long_mbest(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t num, int32_t pmin, int32_t pmax,
                  int32_t gamma, int32_t trunc, int32_t orth, const int32_t *chain_off, const int32_t *chain_q,
                  const int32_t *fac_off, const int32_t *fac, int32_t table_pmax, uint32_t *periods, double *powers,
                  double *bases, int32_t *sweeps, int32_t *near_ties, int32_t *status, void *workspace,
                  size_t workspace_bytes, void *stream);
int pp_long_small_to_large(const double *x, int64_t ldx, int32_t B, int32_t N, double thresh, int32_t n_periods,
                           int32_t trunc, int32_t orth, const int32_t *chain_off, const int32_t *chain_q,
                           int32_t table_pmax, int32_t kmax, uint32_t *periods, double *powers, double *bases,
                           int32_t *count, int32_t *status, void *workspace, size_t workspace_bytes, void *stream);
int pp_long_best_correlation(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t num, int32_t max_length,
                             double ratio, int32_t trunc, int32_t orth, const int32_t *chain_off,
                             const int32_t *chain_q, int32_t table_pmax, uint32_t *periods, double *powers,
                             double *bases, int32_t *status, void *workspace, size_t workspace_bytes, void *stream);
int pp_long_best_frequency_round(double *work, int32_t B, int32_t N, const double *mags, int32_t F, int32_t win_size,
                                 int32_t trunc, int32_t orth, const int32_t *chain_off, const int32_t *chain_q,
                                 int32_t table_pmax, uint32_t *periods, double *norms, double *bases, int32_t round,
                                 int32_t num, int32_t *status, void *workspace, size_t workspace_bytes, void *stream);

/* ---- QOPeriods.find_periods, default branch (QOPeriods.py:313-643, 743-852) ---------------
 * Per window up to `num` rounds: gamma-norm sweep of the residual over [pmin, pmax]
 * (trunc = the instance's trunc_to_integer_multiple, orthogonalize False, :470-478); dictionary
 * rows per period = sum of phi over newly seen divisors (:830-840, a repeated period gets 0 and
 * then contributes all its rows, :972); normal equations against the ORIGINAL data (:781-794);
 * residual = data - reconstruction; stop when rms(reconstruction) <= rms(data) * thresh (:391), in
 * which case the last period is not reported (:585-588).
 *
 * Normal equations.  G = A A^T is integer valued and never stored: its entries have a closed form
 * (Chinese remainder theorem) evaluated where the factorisation consumes them.  The Cholesky factor
 * (reference: LU, np.linalg.solve) is computed left-looking on the FP64 tensor cores (mma.sync m8n8k4,
 * SASS DMMA), packed by block rows, for ANY number of dictionary rows R <= N; `refine` steps of
 * iterative refinement with the implicit Gram product (W - G w = A (x - A^T w): a fold of the signal
 * residual) follow.  R > N makes the system singular by rank (status PP_STATUS_SINGULAR, as a
 * non-positive pivot does: the reference raises LinAlgError or returns rounding noise there); a window
 * with R > rmax reports PP_STATUS_TOO_LARGE (rows needed in n_weights) and keeps the previous round's
 * outputs, so the caller can re-run just those windows (`order`) with a larger rmax.
 *
 * Workspace: pp_qo_workspace_bytes(N, pmax, num, rmax, ctas, basis) holds the factors of `ctas` concurrent windows
 * (0 = one per CTA of the full persistent grid); a smaller workspace only lowers the number of CTAs launched.
 * order (nullable): n_order window indices to process instead of all B (outputs stay indexed by window).
 * phi: device int32 table of Euler's totient for 0..table_pmax.
 * Outputs: periods u32[B,num] (found order, duplicates possible), norms f64[B,num], n_periods[B];
 * dictionary dict_q/dict_keep i32[B,num] in insertion order with n_dict[B]; weights f64[B,ldw]
 * (ldw >= rmax rounded up to 32) with n_weights[B]; res f64[B,N] (nullable); status[B].
 * weights_pool (nullable, natural basis): decouples the size of the dense weights array from rmax.  With a pool, ldw
 * may be smaller than rmax: a window whose dictionary outgrows ldw rows writes its weights to one slot of
 * weights_pool[pool_slots, rmax rounded up to 32] instead, pool_slot[b] = the slot (else -1); a window that finds the
 * pool exhausted reports PP_STATUS_TOO_LARGE.  (Config 5: 1 % of the windows need more than 1024 rows; with the
 * factor storage sized for 2560 rows and a pool for their weights they are solved in the first launch instead of a
 * second one that is bound by its single largest window.) */
/* basis (QOPeriods(basis_type=...), QOPeriods.py:153-155, 940-974):
 *   PP_BASIS_NATURAL    rows 1[n = i (mod q)] (default; Cholesky on the FP64 tensor cores as described above)
 *   PP_BASIS_RAMANUJAN  rows c_q((n - i) mod q) (QOPeriods.py:970-971, 1005-1052).  The q shifted rows of a period span
 *       only phi(q) dimensions, so G is singular by construction; the reference's LU of the rounding-perturbed matrix
 *       yields a reconstruction equal to the orthogonal projection onto the row space (to 1e-14, measured), which is
 *       computed here by conjugate gradients with the rows applied implicitly (folds and circular correlations).
 *       Periods, dictionary, norms and residual match the reference; the weights are the minimum-norm solution (the
 *       reference's are one arbitrary solution of a singular system).  rmax is then only the capacity of `weights`
 *       (rows <= sum of the periods); a window that does not converge reports PP_STATUS_GUARD. */
#define PP_BASIS_NATURAL 0
#define PP_BASIS_RAMANUJAN 1
size_t pp_qo_workspace_bytes(int32_t N, int32_t pmax, int32_t num, int32_t rmax, int32_t ctas, int32_t basis);
int pp_qo_find_periods(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t num, double thresh,
                       int32_t pmin, int32_t pmax, int32_t trunc, int32_t fold_mode, int32_t refine, int32_t basis,
                       const int32_t *phi, int32_t table_pmax, int32_t rmax, const int32_t *order,
                       int32_t n_order, uint32_t *periods, double *norms, int32_t *n_periods, int32_t *dict_q,
                       int32_t *dict_keep, int32_t *n_dict, int32_t *n_weights, double *weights, int64_t ldw,
                       double *res, int32_t *status, double *weights_pool, int32_t pool_slots, int32_t *pool_slot,
                       void *workspace, size_t workspace_bytes, void *profile, void *stream);

/* ---- get_subspaces + solve_quadratic for given periods (QOPeriods.py:743-852; used by
 *      RamanujanPeriods.find_periods_with_weights, RamanujanPeriods.py:106-112) ---------------
 * periods i32[B,kmax] with nper[B] valid entries each, in the caller's order.  weights of window b go to
 * weights + weights_off[b] when weights_off is given (a ragged layout sized by pp_qo_dictionary_rows),
 * else to weights + b * ldw.  A window that is not solved (PP_STATUS_SINGULAR / PP_STATUS_TOO_LARGE) gets res = x. */
int pp_qo_solve(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t *periods,
                const int32_t *nper, int32_t pmax, int32_t refine, const int32_t *phi, int32_t table_pmax,
                int32_t rmax, const int32_t *order, int32_t n_order, int32_t *dict_q, int32_t *dict_keep,
                int32_t *n_dict, int32_t *n_weights, double *weights, int64_t ldw, const int64_t *weights_off,
                double *res, int32_t *status, void *workspace, size_t workspace_bytes, void *stream);

/* The same solve stage for QOPeriods(basis_type="ramanujan") (QOPeriods.py:970-971, 1005-1052): same arguments and
 * outputs as pp_qo_solve, rows c_q((n - i) mod q), the reconstruction computed by conjugate gradients as in
 * pp_qo_find_periods with PP_BASIS_RAMANUJAN (weights: the minimum-norm solution; rmax is only the capacity of
 * `weights`, rows <= sum of the periods).  Periods must lie in [1, pmax].  Status: PP_STATUS_SINGULAR when the
 * dictionary holds both rows of period 2 (the one exact singularity of this basis, where the reference's LU raises),
 * PP_STATUS_TOO_LARGE with the rows needed in n_weights when they exceed rmax, PP_STATUS_GUARD when conjugate
 * gradients do not converge; a window that is not solved gets res = x.  Workspace: pp_qo_workspace_bytes(N, pmax,
 * kmax, rmax, ctas, PP_BASIS_RAMANUJAN); fit query: PP_QO_KIND_SOLVE_RAMANUJAN. */
int pp_qo_solve_ramanujan(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t *periods,
                          const int32_t *nper, int32_t pmax, int32_t refine, const int32_t *phi, int32_t table_pmax,
                          int32_t rmax, const int32_t *order, int32_t n_order, int32_t *dict_q, int32_t *dict_keep,
                          int32_t *n_dict, int32_t *n_weights, double *weights, int64_t ldw, const int64_t *weights_off,
                          double *res, int32_t *status, void *workspace, size_t workspace_bytes, void *stream);

/* rows[b] = rows of the dictionary get_subspaces (QOPeriods.py:830-840) lays out for periods[b, 0:nper[b]):
 * lets the caller size rmax, the ragged weights array and the workspace before pp_qo_solve. */
int pp_qo_dictionary_rows(int32_t B, int32_t kmax, const int32_t *periods, const int32_t *nper, int32_t pmax,
                          const int32_t *phi, int32_t table_pmax, int32_t *rows, void *stream);

/* Solve stage for a caller-supplied dictionary layout: entry k of window b is the period dict_q[b,k] with its
 * first dict_rows[b,k] natural-basis rows (0 = all rows).  Replaces get_subspaces + solve_quadratic of the
 * QOPeriodsWithGCDsExtracted subclass (QOPeriodsWithGCDsExtracted.py:98-143, QOPeriods.py:743-805), whose
 * layout depends on CPython set order and is therefore built by the host layer.  weights[B, ldw],
 * res[B, N] (nullable), status: PP_STATUS_OK / SINGULAR / TOO_LARGE. */
int pp_qo_solve_rows(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t *dict_q,
                     const int32_t *dict_rows, const int32_t *n_dict, int32_t pmax, int32_t refine, int32_t rmax,
                     int32_t *n_weights, double *weights, int64_t ldw, double *res, int32_t *status,
                     void *workspace, size_t workspace_bytes, void *stream);

/* ---- QOPeriods on windows that do not fit in shared memory (the "long" path, pp_long_qo.cu) ----------------
 * pp_qo_fits_on_chip answers, without touching a device, whether the on-chip launch of `kind` fits smem_bytes of
 * shared memory per block.  It evaluates the plan the launch itself would use:
 *   PP_QO_KIND_FIND     pp_qo_find_periods (num, rmax, basis; fold_mode decides the hierarchical scratch: pass
 *                       PP_FOLD_DIRECT for a trunc call, which always folds directly);
 *   PP_QO_KIND_SOLVE    pp_qo_solve / pp_qo_solve_rows (num = kmax; basis must be PP_BASIS_NATURAL), including the
 *                       choice to read the window in place from global memory;
 *   PP_QO_KIND_SOLVE_RAMANUJAN  pp_qo_solve_ramanujan (num = kmax; basis must be PP_BASIS_RAMANUJAN), the same choice;
 *   PP_QO_KIND_MURESAN  pp_muresan_powers (pmax = max_p; num, rmax, basis, fold_mode are checked but unused).
 * Windows or periods above 32767 samples never fit (the on-chip find and solve reject them).  1 = fits, 0 = does
 * not, < 0 = bad arguments.
 * pp_long_qo_find_periods, pp_long_qo_solve, pp_long_qo_solve_ramanujan, pp_long_qo_solve_rows and
 * pp_long_muresan_powers take the arguments of their on-chip namesakes (find: without fold mode, order list, overflow
 * pool and profile buffer; weights are dense, ldw >= rmax rounded up to 32) plus a workspace, and return the same
 * results for any N.  The windows' residuals
 * and each window's packed Cholesky factor live in the workspace; batches run in pieces of windows, as many as the
 * workspace holds (pp_long_qo_workspace_bytes sizes it for a piece of at most half the L2 cache in residuals and at
 * most factor_budget bytes of factors; kind and basis as for pp_qo_fits_on_chip, PP_QO_KIND_SOLVE also accepts
 * PP_BASIS_RAMANUJAN there, which sizes the same per-window state as PP_QO_KIND_SOLVE_RAMANUJAN).  For the Ramanujan
 * basis the conjugate-gradient vectors take the place of the factor.  A dictionary holds at most
 * pp_long_qo_max_rows(smem_bytes) rows (the right-hand side stays in shared memory); above that, and above rmax, a window reports PP_STATUS_TOO_LARGE with the
 * rows it needs in n_weights.  The calls return after their work is done. */
#define PP_QO_KIND_FIND 0
#define PP_QO_KIND_SOLVE 1
#define PP_QO_KIND_MURESAN 2
#define PP_QO_KIND_SOLVE_RAMANUJAN 3
int pp_qo_fits_on_chip(int32_t kind, int32_t N, int32_t pmax, int32_t num, int32_t rmax, int32_t basis,
                       int32_t fold_mode, int32_t smem_bytes);
int32_t pp_long_qo_max_rows(int32_t smem_bytes);
size_t pp_long_qo_workspace_bytes(int32_t kind, int32_t B, int32_t N, int32_t pmax, int32_t num, int32_t rmax,
                                  int32_t basis, size_t factor_budget);
int pp_long_qo_find_periods(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t num, double thresh,
                            int32_t pmin, int32_t pmax, int32_t trunc, int32_t refine, int32_t basis, const int32_t *phi,
                            int32_t table_pmax, int32_t rmax, uint32_t *periods, double *norms, int32_t *n_periods,
                            int32_t *dict_q, int32_t *dict_keep, int32_t *n_dict, int32_t *n_weights, double *weights,
                            int64_t ldw, double *res, int32_t *status, void *workspace, size_t workspace_bytes,
                            void *stream);
int pp_long_qo_solve(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t *periods,
                     const int32_t *nper, int32_t pmax, int32_t refine, const int32_t *phi, int32_t table_pmax,
                     int32_t rmax, const int32_t *order, int32_t n_order, int32_t *dict_q, int32_t *dict_keep,
                     int32_t *n_dict, int32_t *n_weights, double *weights, int64_t ldw, const int64_t *weights_off,
                     double *res, int32_t *status, void *workspace, size_t workspace_bytes, void *stream);
int pp_long_qo_solve_ramanujan(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t *periods,
                               const int32_t *nper, int32_t pmax, int32_t refine, const int32_t *phi, int32_t table_pmax,
                               int32_t rmax, const int32_t *order, int32_t n_order, int32_t *dict_q, int32_t *dict_keep,
                               int32_t *n_dict, int32_t *n_weights, double *weights, int64_t ldw,
                               const int64_t *weights_off, double *res, int32_t *status, void *workspace,
                               size_t workspace_bytes, void *stream);
int pp_long_qo_solve_rows(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t kmax, const int32_t *dict_q,
                          const int32_t *dict_rows, const int32_t *n_dict, int32_t pmax, int32_t refine, int32_t rmax,
                          int32_t *n_weights, double *weights, int64_t ldw, double *res, int32_t *status,
                          void *workspace, size_t workspace_bytes, void *stream);
int pp_long_muresan_powers(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t max_p, int32_t normalize,
                           const int32_t *mu, int32_t table_pmax, double *raw, double *pows, int32_t *best,
                           void *workspace, size_t workspace_bytes, void *stream);

/* ---- QOPeriods.get_periods (QOPeriods.py:719-741 with concatenate_periods :854-887 and
 *      stack_pairwise_gcd_subspaces :889-938), batched ------------------------------------------------------
 * Window b: dictionary entries dict_q[b, 0:n_dict[b]) with dict_keep[b, k] weights each (as pp_qo_find_periods /
 * pp_qo_solve return them; weights at weights + weights_off[b], or + b * ldw when weights_off is null).  The
 * weights are zero padded to one period each and concatenated (sum of q entries); out + out_off[b] receives that
 * vector minus its orthogonal projection onto the row space of the pairwise-GCD matrix (+-comb rows of every
 * pair's gcd, all shifts) -- what every decomp_type of the reference computes ("row reduction", "lu", "qr" and
 * lstsq differ only in how they get rid of the dependent rows).  Conjugate gradients on the normal equations with
 * the rows applied implicitly; iters[b] = steps taken.  tmax / rmax: the largest sum of q and the largest number
 * of rows (sum of the pairs' gcds) in the batch; 2 * tmax + 3 * rmax doubles must fit in shared memory.
 * status: PP_STATUS_OK, PP_STATUS_GUARD (not converged), PP_STATUS_TOO_LARGE (window exceeds tmax / rmax). */
int pp_qo_get_periods(int32_t B, int32_t kmax, int32_t tmax, int32_t rmax, const int32_t *dict_q,
                      const int32_t *dict_keep, const int32_t *n_dict, const double *weights, int64_t ldw,
                      const int64_t *weights_off, double *out, const int64_t *out_off, int32_t *iters,
                      int32_t *status, void *stream);

/* ---- QOPeriods.get_best_period_orthogonal / eq_3 (QOPeriods.py:1122-1232): Muresan's equation-3 finder ----
 * raw[b, q] = eq_3(x_b, q) for q in [1, max_p) (raw[b, 0] = 0; the finder uses max(raw, 0)), with eq_3 evaluated as
 * (q / N) * (energy of the residue-class fold - 2 * autocorrelation at lag (N // q) * q) -- the same quantity as the
 * reference's sum of autocorrelations at multiples of q (:1123-1150);  pows[b, q] = raw minus the powers of the
 * proper divisors (a Moebius inversion of the reference's sequential subtraction, :1209-1217), negatives clamped,
 * divided by q when `normalize`;  best[b] = first arg-max of pows, or 1 when all powers are zero (:1226-1232).
 * raw / pows are nullable, [B, max_p] row-major.  mu: device int32 Moebius table for 0..table_pmax. */
int pp_muresan_powers(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t max_p, int32_t normalize,
                      const int32_t *mu, int32_t table_pmax, double *raw, double *pows, int32_t *best, void *stream);

/* ---- RamanujanPeriods.find_periods (RamanujanPeriods.py:67-86, 124-169) ------------------
 * norms[b, q] = sum_n (sum_i <x, r_i> r_i)[n]^2 over the q-row Ramanujan dictionary of period q,
 * evaluated in fp64 as the dense contraction (q / phi(q)^2) * circ(c_q) * S_q on the FP64 tensor
 * cores (DMMA), S_q = residue-class fold of the window, followed by the count-weighted column
 * norms.  One fused kernel: a CTA folds 16 windows at period q into shared memory and contracts in
 * place; the folds never reach HBM (traffic: the windows once per L2 group, one norm per period).
 * (The reference stores its projection in float32, :127, so its own norms carry ~1e-7
 * relative noise; this path is the fp64 value -- see pp_ramanujan_norms_f32compat for the reference's
 * own numbers.)  mu / phi: device int32 tables (Moebius, totient) for 0..table_qmax.  Only columns
 * qmin..qmax of norms[B, ld_norms] are written.  tile_windows: for PP_RAM_FP64 the number of windows
 * whose samples should stay L2-resident while every period passes over them (1024 = 32 MB at N = 4096);
 * for the other modes the number of windows whose folds the workspace holds at once. */
#define PP_RAM_FP64 0
#define PP_RAM_TF32 1
#define PP_RAM_F32COMPAT 2
size_t pp_ramanujan_workspace_bytes(int32_t N, int32_t qmin, int32_t qmax, int32_t tile_windows, int32_t mode);
int pp_ramanujan_norms(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t qmin, int32_t qmax,
                       const int32_t *mu, const int32_t *phi, int32_t table_qmax, int32_t tile_windows,
                       double *norms, int32_t ld_norms, void *workspace, size_t workspace_bytes, void *stream);

/* TF32 option of the same periodogram on the 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulator in
 * tensor memory, fp32 accumulation): the Ramanujan sums are exact in TF32, the fold sums are split into hi + lo
 * parts; norms agree with the fp64 path to ~1e-5 relative.  The fold itself stays fp64. */
int pp_ramanujan_norms_tf32(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t qmin, int32_t qmax,
                            const int32_t *mu, const int32_t *phi, int32_t table_qmax, int32_t tile_windows,
                            double *norms, int32_t ld_norms, void *workspace, size_t workspace_bytes, void *stream);

/* float32-compat option: the reference's OWN numbers.  RamanujanPeriods.project stores each projected row in a
 * float32 array (RamanujanPeriods.py:127-130); find_periods adds the q rows in float32 in row order (np.sum over
 * axis 0, :77) and sums the squares of the N float32 samples with numpy's pairwise summation (:78).  This entry
 * reproduces that arithmetic operation by operation on top of the fp64 tensor-core products (<x, r_i> in fp64, each
 * product rounded to float32 once, sequential float32 row sum, numpy's 8-lane / 128-block pairwise tree), so the
 * norms equal the reference's to the last float32 bit except where the reference's own 1e-13 noise in Cq
 * (:142-144, a sum of complex exponentials) moves a rounding.  Workspace: pp_ramanujan_workspace_bytes with
 * PP_RAM_F32COMPAT (the products H S_q of a tile are kept beside its folds).  N <= 32768. */
int pp_ramanujan_norms_f32compat(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t qmin, int32_t qmax,
                                 const int32_t *mu, const int32_t *phi, int32_t table_qmax, int32_t tile_windows,
                                 double *norms, int32_t ld_norms, void *workspace, size_t workspace_bytes,
                                 void *stream);

/* pp_ramanujan_fits_on_chip answers, without touching a device, whether the on-chip launch of `mode` (PP_RAM_*) fits
 * smem_bytes of shared memory per block.  It evaluates the plan the launch itself uses: the fused kernel for
 * PP_RAM_FP64; the fold, contraction and tcgen05 / compat kernels, and N <= 32768 for PP_RAM_F32COMPAT, for the
 * others.  1 = fits, 0 = does not, -1 = bad arguments.  An fp64 periodogram that does not fit can be computed by
 * pp_ramanujan_norms_divisor, for any N. */
int pp_ramanujan_fits_on_chip(int32_t mode, int32_t N, int32_t qmin, int32_t qmax, int32_t smem_bytes);

/* ---- the Ramanujan periodogram in divisor form (pp_ram_divisor.cu) ---------------------------------------------
 * The same fp64 quantity as pp_ramanujan_norms (PP_RAM_FP64), computed without the dense contraction:
 * c_q(n) = sum_{d | gcd(n, q)} mu(q/d) d turns H S_q into an in-place product over the distinct primes p of q,
 *     z = (q / rad(q)) prod_p (p I - A_p) S_q,     (A_p v)_m = sum_{k < p} v[(m + k q / p) mod q],
 * and norms[b, q] = (q / phi(q)^2)^2 sum_m cnt_q[m] z_m^2.  Work per (window, period): the fold (N adds, summed in
 * increasing n per residue as the sweeps do) plus about 2 omega(q) q; no dense product, so the norms differ from the
 * dense path's by rounding only (rtol 1e-11).  Each (window, period) is computed by one warp or one CTA with
 * fixed-order sums: two runs are bit-identical.
 * staging: PP_STAGING_SHARED stages each window in shared memory once and spreads its periods over the CTA's warps
 * (fails with -1 when that plan does not fit the device); PP_STAGING_GLOBAL folds every (window, period) unit from
 * global memory (L2), any N; PP_STAGING_AUTO takes SHARED when the plan fits.
 * pp_ramanujan_divisor_fits_on_chip answers, without touching a device, whether the SHARED plan fits smem_bytes of
 * shared memory per block: 1 / 0, -1 on bad arguments.
 * pp_ramanujan_divisor_workspace_bytes: a 256-byte unit counter plus, when qmax > 8192, one scratch slice of
 * qmax + ceil(qmax / 2) doubles (+ 1, rounded to even) per CTA of the global-memory launch (at most 296), i.e. at most
 *     256 + 296 * 8 * (qmax + ceil(qmax / 2) + 2) bytes  (O(CTAs x qmax), nothing grows with qmax^2);
 * 0 on bad arguments.  A smaller workspace lowers the number of CTAs the global-memory launch uses.
 * spf / phi: device int32 tables (smallest prime factor, totient) for 0..table_qmax.  Only columns qmin..qmax of
 * norms[B, ld_norms] are written. */
#define PP_STAGING_AUTO 0
#define PP_STAGING_SHARED 1
#define PP_STAGING_GLOBAL 2
int pp_ramanujan_divisor_fits_on_chip(int32_t N, int32_t qmin, int32_t qmax, int32_t smem_bytes);
size_t pp_ramanujan_divisor_workspace_bytes(int32_t B, int32_t N, int32_t qmin, int32_t qmax);
int pp_ramanujan_norms_divisor(const double *x, int64_t ldx, int32_t B, int32_t N, int32_t qmin, int32_t qmax,
                               const int32_t *spf, const int32_t *phi, int32_t table_qmax, int32_t staging,
                               double *norms, int32_t ld_norms, void *workspace, size_t workspace_bytes, void *stream);

/* periods[b, 0:nper[b]] = ascending q in [0, qlen) with norms[b,q] / |max_q norms[b,q]| > thresh
 * (RamanujanPeriods.py:97-101); nper[b] may exceed kmax, only the first kmax are stored. */
int pp_ramanujan_select(const double *norms, int32_t B, int32_t ld_norms, int32_t qlen, double thresh,
                        int32_t kmax, int32_t *periods, int32_t *nper, void *stream);

/* ---- the one collective of the path (SURVEY.md 8e): gather of compact results over NCCL / NVLink ---------
 * Windows shard across GPUs with no data-path exchange; only the compact outputs (periods u32, powers f64, status
 * i32: ~124 B per window) travel to one rank.  pp_gather enqueues that exchange on `stream` -- the compute stream,
 * right behind the last kernel, no host synchronisation -- as ncclGather (NCCL >= 2.28) or the equivalent grouped
 * ncclSend / ncclRecv.  Every rank sends `bytes` bytes; `recv` (root only, nranks * bytes) receives them in rank order.
 * NCCL is resolved at run time (dlopen of the libnccl.so.2 already in the process, or the path given to
 * pp_comm_load); the library has no link-time dependency on it.  Communicator bootstrap: rank 0 calls
 * pp_comm_unique_id and hands the 128 bytes to the other ranks by any channel (the Python layer broadcasts them
 * with torch.distributed), then every rank calls pp_comm_init. */
int pp_comm_load(const char *library_path);        /* optional: explicit path of libnccl.so.2 */
int pp_comm_version(void);                         /* NCCL version code (e.g. 22809), -1 if NCCL is unavailable */
int pp_comm_unique_id(void *id_out_128_bytes);
int pp_comm_init(void **comm_out, int32_t nranks, int32_t rank, const void *id_128_bytes);
int pp_comm_destroy(void *comm);
int pp_gather(void *comm, const void *send, void *recv, size_t bytes, int32_t root, void *stream);

/* ---- roofline denominators measured live (BASELINE.md section 3) -----------------------
 * kind 0: shared-memory load bandwidth, out_host[0] = bytes/s over the whole chip;
 * kind 1: FP64 add throughput,           out_host[0] = adds/s  over the whole chip;
 * kind 2: FP64 tensor cores (DMMA m8n8k4), out_host[0] = flop/s over the whole chip;
 * out_host[1] = SM clock (MHz) observed during the run, out_host[2] = kernel ms.
 * Synchronous; allocates and frees its own 64-byte scratch. */
int pp_microbench(int32_t kind, int32_t iters, double *out_host);

#ifdef __cplusplus
}
#endif
#endif /* PYPERIOD_B200_H */
