/* sbo_b200.h -- C ABI of the B200-native SafeOpt/GoOSE grid hot path.
 *
 * Drop-in boundary for the ONE data-parallel path of dleeim/Safe-Bayesian-Optimization:
 * per acquisition step, GP posteriors over a dense candidate grid, then the safe set,
 * minimiser set, expander set / GoOSE target and the arg-reductions that pick x_new.
 * The reference has no native code and no FFI; each entry point below cites the
 * reference *Python* interface it replaces (paths relative to the reference root).
 * Python binds this library with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - every function returns 0 on success, a negative sbo_status otherwise; the message
 *     is available from sbo_last_error().  Nothing aborts.  There is NO CPU fallback: a
 *     context cannot be created without a CUDA device.
 *   - host pointers unless the name ends in _dev.  The caller owns all in/out buffers;
 *     the context owns device copies, workspaces and (unless sbo_set_stream) its stream.
 *   - calls are synchronous w.r.t. returned host data; one host thread per context.
 *   - all floating-point data is FP64 (the reference runs jax_enable_x64, GP_Safe.py:8).
 *   - grid points are numbered with x_0 the fastest axis (test/test_SafeOpt.py:324-334:
 *     meshgrid 'xy' + ravel  =>  p = r*400 + c).  Indices returned are GLOBAL grid
 *     indices (int64); -1 means "empty set".
 *   - per-point arrays are GP-major: mean[i*count + p], i = GP index (0 = objective).
 *   - bitmasks are little-endian uint32 words over the LOCAL shard: bit (p&31) of word p>>5.
 */
#ifndef SBO_B200_H
#define SBO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SBO_MAX_D 8   /* input dimensions  */
#define SBO_MAX_G 8   /* GPs: 1 objective + up to 7 constraints */

typedef struct sbo_ctx sbo_ctx;

enum sbo_status {
  SBO_OK = 0,
  SBO_ERR_INVALID = -1,   /* bad argument / call order  */
  SBO_ERR_CUDA = -2,      /* CUDA runtime error         */
  SBO_ERR_NUMERIC = -3,   /* K not positive definite    */
  SBO_ERR_NOMEM = -4
};

/* unsafe-set rule.  ALL: Z = {z : lcb_i(z) <= 0 for every constraint}  -- what the reference's
 * lcb_constraint_min (returns the MAX, models/SafeOpt.py:73-77) + "<= 0" (SafeOpt.py:109) encodes.
 * ANY: Z = {z : some lcb_i(z) < 0} = complement of S. */
enum sbo_unsafe_rule { SBO_UNSAFE_ALL = 0, SBO_UNSAFE_ANY = 1 };

enum sbo_expander_mode { SBO_MODE_LIPSCHITZ = 0, SBO_MODE_FANTASY = 1 };

/* covariance function of a model (sbo_set_model_ex, sbo_nll_batch_ex).  With the scaled squared distance
 * s = sum_k (x_k - x'_k)^2 / ell_k of the ARD hyper-parameters:
 *   SE        k = sf2 exp(-s/2)                      (GP_Safe.py:98-120, the reference's 'RBF')
 *   MATERN32  k = sf2 (1 + t) exp(-t),        t = sqrt(3 s)
 *   MATERN52  k = sf2 (1 + t + t^2/3) exp(-t), t = sqrt(5 s)
 * Every GP of a model uses the same kernel; k(x, x) = sf2 for all three. */
enum sbo_kernel { SBO_KERNEL_SE = 0, SBO_KERNEL_MATERN32 = 1, SBO_KERNEL_MATERN52 = 2 };
enum sbo_precision { SBO_PREC_FP64 = 0, SBO_PREC_TF32 = 1, SBO_PREC_TF32X3 = 2 };

/* score selectors for sbo_argreduce */
enum sbo_reduce_kind {
  SBO_ARGMAX_VAR0 = 0,     /* max objective variance over a mask        (SafeOpt.py:55,65,92) */
  SBO_ARGMIN_LCB0 = 1,     /* min lcb_0 over a mask                     (GoOSE.py:63-67,110)  */
  SBO_ARGMIN_UCB0 = 2,     /* min ucb_0 over a mask                     (SafeOpt.py:47-51)    */
  SBO_ARGMIN_DIST = 3      /* min ||x - target||_2 over a mask          (GoOSE.py:116-119)    */
};
enum sbo_mask_kind { SBO_MASK_SAFE = 0, SBO_MASK_MIN = 1, SBO_MASK_UNSAFE = 2, SBO_MASK_USER = 3 };

/* ---- lifetime ------------------------------------------------------------------------ */
int sbo_create(int device, sbo_ctx** out);
int sbo_destroy(sbo_ctx* ctx);
const char* sbo_last_error(const sbo_ctx* ctx);        /* ctx may be NULL: last create() error */
int sbo_set_stream(sbo_ctx* ctx, void* cuda_stream);   /* run on the caller's stream (e.g. torch's) */
int sbo_version(void);

/* ---- model upload:  GP.inference_datasets  (models/GP_Safe.py:16-23,236-245) ------------
 * X_norm[n*d] row-major, Y_norm[n*G] row-major, hyp[(d+2)*G] row-major with rows
 * [0:d] = 1/2 log ell, [d] = 1/2 log sf2, [d+1] = 1/2 log sn2  (GP_Safe.py:226-229).
 * Builds K_i = sf2*exp(-1/2 dist) + (sn2 + eps_f32) I  (GP_Safe.py:229-231) on the device,
 * factorises it (K = L L^T), forms W = L^-1 and alpha = K^-1 (Y_i - m0_i) with the
 * reference's prior mean m0 = -2*Y_mean/Y_std, m0[0] = 0  (GP_Safe.py:331-332).
 * Replaces jnp.linalg.inv(Kopt) (GP_Safe.py:232): the explicit inverse is never needed. */
int sbo_set_model(sbo_ctx* ctx, int n, int d, int G,
                  const double* X_norm, const double* Y_norm,
                  const double* X_mean, const double* X_std,
                  const double* Y_mean, const double* Y_std,
                  const double* hyp);
/* sbo_set_model with the covariance function `kernel` (enum sbo_kernel) in place of the SE kernel: K_i = k_i(X, X) + (sn2 +
 * eps_f32) I with the same hyper-parameter layout.  sbo_set_model is the SBO_KERNEL_SE case.  The kernel stays part of the
 * installed model: sbo_append_sample, the posterior, the sets, every pair test and the sharded steps use it.  The separable
 * options "posterior_tables" and "posterior_fused" exist for the SE kernel only and are ignored for the others. */
int sbo_set_model_ex(sbo_ctx* ctx, int kernel, int n, int d, int G,
                     const double* X_norm, const double* Y_norm,
                     const double* X_mean, const double* X_std,
                     const double* Y_mean, const double* Y_std,
                     const double* hyp);
/* One more observation at FIXED hyper-parameters and FIXED normalisation (SURVEY.md section 8f row 1): x_norm_new[d],
 * y_norm_new[G] in the normalised units of the installed model.  Rank-1 update of the factor on the device -- new row of
 * L, of W = L^-1 and a refreshed alpha, O(n^2) -- instead of the rebuild + O(n^3) inverse of GP.add_sample
 * (models/GP_Safe.py:283-304, which also re-fits and re-normalises; use sbo_set_model for that semantics). */
int sbo_append_sample(sbo_ctx* ctx, const double* x_norm_new, const double* y_norm_new);
/* debug / test read-back (any pointer may be NULL): K,L,W are [G][n][n] row-major, alpha [G][n] */
int sbo_get_model(sbo_ctx* ctx, double* L, double* W, double* alpha);

/* ---- candidate points:  create_data_for_plot()  (test/test_SafeOpt.py:324-334) ---------
 * sbo_set_grid: implicit meshgrid of per-axis numpy.linspace(lo_k, hi_k, pts_k), x_0 fastest.
 * sbo_set_points: explicit N x d row-major points.
 * sbo_set_shard: this context (rank) owns global points [first, first+count); default = all. */
int sbo_set_grid(sbo_ctx* ctx, int d, const int64_t* pts_per_dim, const double* lo, const double* hi);
int sbo_set_points(sbo_ctx* ctx, int64_t N, int d, const double* pts);
int sbo_set_shard(sbo_ctx* ctx, int64_t first, int64_t count);
/* rotated block-cyclic ownership (multi-GPU): the grid is cut into blocks of `block` consecutive points (a
 * multiple of 32); in super-block sb (nranks consecutive blocks) rank r owns slot (r + sb + sb/nranks +
 * sb/nranks^2) % nranks, which balances |S| and |Z| across ranks even when the meshgrid axes are multiples of
 * block*nranks.  Local point p (sb = p / block) maps to global index (sb*nranks + slot)*block + p % block;
 * *count = number of local points. */
int sbo_set_shard_cyclic(sbo_ctx* ctx, int rank, int nranks, int64_t block, int64_t* count);
int sbo_point_coords(sbo_ctx* ctx, int64_t global_idx, double* x /* d */);

/* ---- posterior:  GP.GP_inference vmapped over the grid  (GP_Safe.py:310-352) -------------
 * mean/var: [G*count] GP-major, raw (un-normalised) units, var clamped >= 0; NULL = keep on device.
 * with_grad != 0 also accumulates L_i = max_p ||grad mu_i(p)||_inf  (SafeOpt.py:68-83).
 * keep_v != 0 keeps V_i = L_i^-1 K_i(X, .) for the fantasy expander (constraints only):
 *   1 = FP64 rows, 2 = FP32 rows rounded to TF32 (tensor-core operand), 3 = split-TF32 rows [hi | lo]
 *   (three-pass TF32 GEMM, ~FP32 accuracy). */
int sbo_posterior(sbo_ctx* ctx, int with_grad, int keep_v, double* mean, double* var);
/* bring the last sbo_posterior of this context up to the model after the sbo_append_sample calls made since (same with_grad,
 * same keep_v); mean/var as in sbo_posterior (NULL = keep on device).  Appending leaves the leading block of L and of
 * W = L^-1 unchanged, so only the m new rows of W enter:  e_r(p) = sum_j W[r][j] k_j(p) for the new rows r,
 * var' = max(0, var/Y_std^2 - sum_r e_r^2) * Y_std^2 per GP, and the kept V rows gain the m columns e(p) (entries of the
 * old rows untouched).  Mean and L_i are recomputed from the new alpha with the loop of sbo_posterior: bitwise what
 * sbo_posterior returns on the same model with the default options.  n kernel values and m*n FMAs per point and GP, no
 * triangular solve; ceil(m/8) kernel launches.  Works on the local shard (contiguous or block-cyclic), no collective.
 *   info->rows = m, the samples appended since; m = 0: nothing to do.  info->recomputed = 1: V rows were kept and the
 *   appends grew the padded factor (the V-row stride changed), so the full sbo_posterior ran with the same flags.
 * SBO_ERR_INVALID, nothing modified: no sbo_posterior since the last sbo_set_model(_ex), sbo_set_grid, sbo_set_points,
 * sbo_set_shard or sbo_set_shard_cyclic, or kept V rows freed by sbo_release(1) since.  Afterwards the sets, pair stages,
 * batches and sbo_lipschitz (with_grad) work as after sbo_posterior. */
typedef struct sbo_update_info { int64_t rows; int32_t recomputed, pad; } sbo_update_info;
int sbo_posterior_update(sbo_ctx* ctx, double* mean, double* var, sbo_update_info* info);
/* GP_inference at m arbitrary points (the single-point API behind BO.mean/ucb/lcb,
 * SafeOpt.py:29-45): x[m*d] row-major -> mean[m*G], var[m*G] POINT-major like the reference. */
int sbo_point_posterior(sbo_ctx* ctx, int64_t m, const double* x, double* mean, double* var);
/* max_p ||grad mu_i||_inf over the local shard, i = 0..G-1 (valid after sbo_posterior(with_grad=1)) */
int sbo_lipschitz(sbo_ctx* ctx, double* L /* G */);
/* d mu_i / d x at m arbitrary points: grad[m*d]  (BO.infnorm_mean_grad's autodiff, SafeOpt.py:68-71) */
int sbo_point_mean_grad(sbo_ctx* ctx, int gp, int64_t m, const double* x, double* grad);

/* ---- sets:  SafeOpt.py:47-66, GoOSE.py:22-31,63-67 -----------------------------------------
 * pass 1: lcb/ucb, S = {lcb_i >= 0 (or > 0 if strict) for all i>=1}, Z by rule,
 *         min_S ucb_0 and argmin_S lcb_0.
 * pass 2: M = {x in S : lcb_0(x) <= min_ucb0} and argmax_M var_0   (SafeOpt.Minimizer).
 * Multi-GPU: all-reduce-min min_ucb0 between the passes and hand the global value to pass 2. */
typedef struct sbo_sets_result {
  int64_t n_safe, n_unsafe, n_min;
  double  min_ucb0;      int64_t min_ucb0_idx;     /* BO.minimize_obj_ucb   */
  double  min_lcb0;      int64_t min_lcb0_idx;     /* BO.minimize_obj_lcb   */
  double  minimizer_var; int64_t minimizer_idx;    /* BO.Minimizer: std = sqrt(var) */
} sbo_sets_result;
int sbo_sets_pass1(sbo_ctx* ctx, double beta, int unsafe_rule, int strict, sbo_sets_result* out);
int sbo_sets_pass2(sbo_ctx* ctx, double min_ucb0, sbo_sets_result* out);
int sbo_sets(sbo_ctx* ctx, double beta, int unsafe_rule, int strict, sbo_sets_result* out);
/* copy a bitmask of the local shard to the host: words[(count+31)/32] */
int sbo_get_mask(sbo_ctx* ctx, int mask_kind, int which, uint32_t* words);
int sbo_set_user_mask(sbo_ctx* ctx, const uint32_t* words);
/* user mask = (mask_kind, e.g. SBO_MASK_SAFE; -1 = all points) AND the ball ||x - x0||_2 <= r, built on the device from the
 * grid coordinates: the feasible set of GP_TR.BO.minimize_obj_lcb (models/GP_TR.py:43-54: safe set within the trust region) */
int sbo_user_mask_ball(sbo_ctx* ctx, int mask_kind, const double* x0 /* d */, double r);
/* device addresses for collectives on the caller's side (NCCL via torch.distributed) */
int sbo_mask_dev(sbo_ctx* ctx, int mask_kind, int which, void** dev_ptr, int64_t* n_words);
int sbo_posterior_dev(sbo_ctx* ctx, void** mean_dev, void** var_dev);

/* ---- arg-reductions (deterministic, lowest-index tie-break): SafeOpt.py:65,112; GoOSE.py:65,102,118 */
int sbo_argreduce(sbo_ctx* ctx, int reduce_kind, int mask_kind, int which, const double* target /* d or NULL */,
                  int64_t* idx, double* value);

/* ---- StableOpt on the grid (models/StableOpt.py:96-160): the meshgrid's first n_controlled axes are x_c, the others
 * the disturbance d.  Robust safe set {x_c : min_d lcb_i(x_c,d) >= 0 for all constraints} (Minimise_d, :147-149),
 * score(x_c) = max_d fun_0(x_c,d) with fun = 0 mean | 1 ucb | 2 lcb (Maximise_d, :151), and the arg-min of the score over
 * the robust safe set (Minimize_Maximise, :153).  xc_idx indexes the x_c sub-grid (x_0 fastest), -1 = empty set;
 * score (optional, host) receives max_d fun_0 for every x_c.  Needs sbo_posterior on the whole, unsharded meshgrid;
 * option "prior_mean_zero" = 1 installs the zero prior mean of GP_Robust.py:322-323 at the next sbo_set_model. */
int sbo_stable_minmax(sbo_ctx* ctx, int n_controlled, int fun_kind, double beta, int64_t* xc_idx, double* value,
                      int64_t* n_robust_safe, double* score);

/* ---- expander / target pair kernels ----------------------------------------------------------
 * Lipschitz mode (reference-exact): pair test  ucb_idx(x) - L_idx*||x - z + 1e-8||_2 >= 0 with
 *   x in S, z in Z  (SafeOpt.py:85-88,109-111; GoOSE.py:69-72,99-101).  L[G]: entry idx is used for
 *   constraint idx (the reference passes L_{G-1} for every idx, SafeOpt.py:110).
 * Fantasy mode (north_star, not in the reference): rank-1 posterior update of every constraint GP with
 *   the observation ucb_i(x); z is newly safe if every updated lcb_i(z) >= 0; g(x) = #newly-safe z.  The fantasy GoOSE
 *   target is T = {z : some x in S makes z newly safe} (a column OR over the same pairs) and its argmin lcb_0.
 *   precision: FP64 (FP64 tensor cores: DMMA mma.sync.m8n8k4.f64 tiles), TF32 (tcgen05/TMEM GEMM, FP32 accumulate) or TF32X3
 *   (same kernel over split operands: x_hi.z_hi + x_hi.z_lo + x_lo.z_hi).
 */
typedef struct sbo_pair_result {
  int64_t best_idx;  double best_value;          /* SafeOpt: argmax var_0 (value = var_0); GoOSE: argmin lcb_0 */
  int64_t per_idx[SBO_MAX_G]; double per_value[SBO_MAX_G];   /* entry idx-1 for constraint idx */
  int64_t n_x, n_z;                              /* candidate / unsafe points paired  */
  int64_t pairs_algorithmic;                     /* n_x * n_z * (constraints)         */
  int64_t pairs_evaluated;                       /* after tile-level early exit       */
  int64_t n_hit;                                 /* |expander set| (union over idx) or |target set| */
  int64_t n_ambiguous, n_refined_safe;           /* fantasy TF32/TF32X3: pairs inside the error bound (re-evaluated in FP64 unless bounds mode) / of those, newly safe;
                                                    GoOSE target: n_refined_safe = unsafe points the FP64 pass added to T (points, not pairs) */
  /* bounds mode ("fantasy_refine" = 3): n_hit counts the candidates with at least one pair SETTLED newly safe (certified members of the
   * FP64 expander set); n_undecided the candidates with no settled pair but at least one pair inside the error bound (the FP64 set is
   * the certified set plus a subset of these); undecided_best_* = argmax var_0 over them (-1 if none).  The reported x_new (best_idx)
   * equals the FP64 one whenever undecided_best_value < best_value.  counts[] then holds the settled counts, -1 for undecided candidates.
   * GoOSE target: n_hit = |certified T| (z with a pair the bound settles as safe); n_undecided = the z not certified with at least one pair
   * inside the bound; undecided_best_* = argmin lcb_0 over them.  The FP64 T is the certified set plus a subset of the undecided z, so
   * best_idx is the FP64 target whenever undecided_best_value > best_value. */
  int64_t n_undecided, undecided_best_idx; double undecided_best_value;
} sbo_pair_result;
int sbo_expander(sbo_ctx* ctx, int mode, int precision, double beta, const double* L /* G, lipschitz mode */,
                 sbo_pair_result* out, int32_t* counts /* count, fantasy mode, or NULL */);
int sbo_goose_target(sbo_ctx* ctx, double beta, const double* L /* G */, sbo_pair_result* out);
/* GoOSE target in either pair test: sbo_goose_target is the Lipschitz case.  Fantasy mode needs sbo_posterior with keep_v as for
 * sbo_expander; the target mask is SBO_MASK_TARGET, which = 0, and the precisions and "fantasy_refine" modes mean what they mean for
 * the expander (fantasy_refine = 2: the TF32 / TF32X3 target set is the FP64 one). */
int sbo_goose_target_ex(sbo_ctx* ctx, int mode, int precision, double beta, const double* L /* G, lipschitz mode */,
                        sbo_pair_result* out);
/* ---- the same pair stage in five steps, for a grid sharded over ranks (SURVEY.md section 8e) ---------------
 * Every rank pairs ALL candidates x in S (gathered from all ranks) with ITS OWN unsafe points z:
 *   sbo_pairs_prepare     compact the local S and Z, build the local z-side operands
 *   sbo_pairs_export_dev  write the local candidates' rows [coords d | ucb G-1 | xn d | a G-1 | b G-1 | grid index] (doubles,
 *                         row_doubles per candidate) and, in fantasy mode, their V rows (vrow_bytes per
 *                         candidate) into caller-owned DEVICE buffers  -> all-gather them (NCCL)
 *   sbo_pairs_import_dev  hand the concatenation of all ranks' rows back (n_total candidates)
 *   sbo_pairs_run_dev     result_dev: lipschitz uint8[(G-1)*n_total] hit flags | fantasy int32[n_total] counts
 *                         (goose: lipschitz uint8[(G-1)*n_z_local] | fantasy uint32[ceil(n_z_local/32)] hit words over the
 *                         prepared, key-sorted unsafe slots; no exchange needed) -> all-reduce max / sum (NCCL)
 *   sbo_pairs_finish_dev  masks + arg-reductions on the local shard; the local candidates are rows
 *                         [offset, offset + n_x_local) of the reduced result.  `out` holds LOCAL optima with
 *                         GLOBAL indices; the caller reduces them across ranks (value, then lowest index).
 * sbo_expander / sbo_goose_target are these five steps on one GPU.  Any model, grid, shard, posterior or sets-pass-1 change
 * invalidates a prepared stage, and sbo_release(1) a fantasy stage's export: the staged calls then fail with SBO_ERR_INVALID. */
typedef struct sbo_pairs_info { int64_t n_x_local, n_z_local, row_doubles, vrow_bytes; } sbo_pairs_info;
int sbo_pairs_prepare(sbo_ctx* ctx, int mode, int precision, double beta, const double* L /* G or NULL */, sbo_pairs_info* info);
int sbo_pairs_export_dev(sbo_ctx* ctx, void* rows_dev, void* vrows_dev);
int sbo_pairs_import_dev(sbo_ctx* ctx, int64_t n_total, const void* rows_dev, const void* vrows_dev);
int sbo_pairs_run_dev(sbo_ctx* ctx, int goose, void* result_dev);
int sbo_pairs_finish_dev(sbo_ctx* ctx, int goose, int64_t offset, const void* result_dev, sbo_pair_result* out, int32_t* counts);
/* Sharded runs, Lipschitz mode (models/SafeOpt.py:85-124 with the grid split over ranks):
 *   sbo_pairs_set_segments           (after prepare) how many candidates every rank exported, and this rank: the gathered
 *                                    rows are put back into grid order inside the library (compact tiles for the exact
 *                                    culling); results stay in the caller's gathered order.
 *   sbo_mask_export_dev              copy a local bitmask into a caller-owned DEVICE buffer (zero padded to dst_words),
 *                                    e.g. the unsafe mask for the all-gather north_star names (N/8 bytes in total).
 *   sbo_pairs_set_global_unsafe_dev  hand the all-gathered local UNSAFE masks back (rank-major, words_per_rank each):
 *                                    the SafeOpt expander then pairs THIS rank's share of the candidate tiles with ALL
 *                                    unsafe points in grid order, so the per-candidate early exit and the tile culling
 *                                    do the same work as on one GPU, divided by the number of ranks.  The per-candidate
 *                                    hit flags are combined with the same all-reduce(max) as before. */
int sbo_pairs_set_segments(sbo_ctx* ctx, int nranks, int rank, const int64_t* n_per_rank);
int sbo_mask_export_dev(sbo_ctx* ctx, int mask_kind, int which, void* dst_dev, int64_t dst_words);
int sbo_pairs_set_global_unsafe_dev(sbo_ctx* ctx, const void* gathered_words_dev, int64_t words_per_rank, int nranks);
/* which = idx-1 (lipschitz/target: one mask per constraint) ; fantasy (expander and target): which = 0 */
#define SBO_MASK_EXPANDER 4
#define SBO_MASK_TARGET   5

/* ---- multi-GPU: library-owned communicator and whole sharded steps (SURVEY.md section 8b/8e) -------------------
 * One process per GPU, one context per process, the grid sharded with sbo_set_shard_cyclic(rank, nranks, block).
 * NCCL is resolved at run time (dlopen libnccl.so.2): no torch / framework needed on the host side.
 *   sbo_comm_unique_id  rank 0 creates the 128-byte ncclUniqueId and distributes it to the other ranks by any host
 *                       mechanism (file, MPI, socket, torch.distributed ...)
 *   sbo_comm_init       collective: every rank joins the communicator
 * sbo_safeopt_step_sharded / sbo_goose_step_sharded run  posterior -> sets -> (Lipschitz constants) -> pair stage ->
 * arg-reductions -> x_new  with the collectives issued on the context's stream between the kernels; every rank gets
 * the same GLOBAL result.  The model must have been installed on every rank (sbo_set_model).  Decision rules:
 * test/test_SafeOpt.py:144-158, test/test_GoOSE.py:151-162.  L = NULL: Lipschitz constants from the grid
 * (SafeOpt.py:68-83), constraint G-1's for every constraint like the reference (SafeOpt.py:110). */
typedef struct sbo_step_result {
  sbo_sets_result sets;            /* global sets: sizes, min_S ucb_0 / lcb_0, minimiser (SafeOpt) */
  double L[SBO_MAX_G];             /* global Lipschitz constants (Lipschitz mode, when computed) */
  sbo_pair_result pairs;           /* expander (SafeOpt) or target (GoOSE): global optima and totals */
  int64_t x_new_idx, explore_idx;  /* chosen next query point (global grid index); GoOSE: nearest safe point or -1 */
} sbo_step_result;
int sbo_comm_unique_id(void* id128);
int sbo_comm_init(sbo_ctx* ctx, int rank, int nranks, const void* id128);
int sbo_comm_destroy(sbo_ctx* ctx);
int sbo_safeopt_step_sharded(sbo_ctx* ctx, double beta, int mode, int precision, int unsafe_rule, const double* L /* G or NULL */,
                             sbo_step_result* out);
int sbo_goose_step_sharded(sbo_ctx* ctx, double beta, int unsafe_rule, const double* L /* G or NULL */, sbo_step_result* out);
/* the GoOSE step in either pair test (sbo_goose_step_sharded is the Lipschitz case).  Fantasy mode: the posterior keeps the V rows of
 * `precision` and computes no gradient (L is ignored); every rank pairs all candidates with its own unsafe points, so the target set
 * needs no result collective. */
int sbo_goose_step_sharded_ex(sbo_ctx* ctx, double beta, int mode, int precision, int unsafe_rule, const double* L /* G or NULL */,
                              sbo_step_result* out);

/* ---- batch SafeOpt acquisition: q safe query points per step (additive; no reference counterpart) -------------------
 * GP-BUCB-style hallucination on the objective GP (index 0), in its normalised units.  The candidates are C = M u E of the
 * last SafeOpt pair stage on the local shard (M = SBO_MASK_MIN; E = the union of its SBO_MASK_EXPANDER masks: Lipschitz mode
 * one per constraint, fantasy mode which = 0, bounds mode the certified members).  S, M and E stay those of the real data,
 * so every pick is in S.  After picks x_1..x_b (hallucinated observations with noise sn = exp(2 hyp[d+1, 0]) + eps_f32,
 * whatever their values) the objective variance is the exact GP posterior variance
 *   v_b(p) = max(0, v_{b-1}(p) - w_b(p)^2),   w_b(p) = (c(p, x_b) - sum_{j<b} R_bj w_j(p)) / R_bb,
 *   c(p, x) = k(p, x) - k(X, p)^T K^-1 k(X, x),   [c(x_i, x_j)] + sn I = R R^T (lower Cholesky, one row per pick),
 * v_0 = the step's var_0.  Pick b uses the decision rule of test/test_SafeOpt.py:153-158 on v_{b-1}: std_M = sqrt(max over M
 * of var_0 in raw units) and std_E the same over E (lowest global index on ties); M's point if std_M > std_E, else E's; a
 * set that is empty yields to the other.  Pick 1 is the step's x_new.  A point may be picked again (what the rule says at
 * noise sn).  A batch reads the step's state and writes none of it: model, posterior, masks and pair results are unchanged.
 * Every entry point needs a SafeOpt pair stage (sbo_expander or a sharded SafeOpt step, with sbo_sets_pass2) since the last
 * model, grid, shard, posterior or set change, and fails with SBO_ERR_INVALID after a GoOSE target stage. */
#define SBO_BATCH_MAX_Q 256   /* picks per batch */
typedef struct sbo_batch_pick {
  int64_t idx;                          /* global index of this pick; -1 = M and E both empty */
  int32_t from_expander, pad;           /* 0: taken from M, 1: from E */
  double  std_min; int64_t idx_min;     /* sqrt(max v * Y_std0^2) over M under the earlier picks (0 / -1 if empty) */
  double  std_exp; int64_t idx_exp;     /* the same over E */
} sbo_batch_pick;
/* one GPU: q picks with no host synchronisation between them (about 3q launches, one copy to the host at the end).
 * picks[q] out; *n_picked = q, or 0 when M and E are both empty (picks[0].idx = -1). */
int sbo_safeopt_batch(sbo_ctx* ctx, int q, sbo_batch_pick* picks, int* n_picked);
/* the same in three steps for a grid sharded over ranks; the batch-side state is computed identically on every rank:
 *   sbo_batch_prepare  compact this rank's candidates, v = var_0 (*n_candidates_local = |C| of the shard)
 *   sbo_batch_local    this rank's optima for the next pick (GLOBAL indices; idx / from_expander apply the rule locally)
 *                      -> the caller reduces (std, index) over the ranks (largest std, lowest index) and applies the rule
 *   sbo_batch_commit   hallucinate an observation at the chosen GLOBAL index (the same on every rank); at most q commits */
int sbo_batch_prepare(sbo_ctx* ctx, int q, int64_t* n_candidates_local);
int sbo_batch_local(sbo_ctx* ctx, sbo_batch_pick* local_optima);
int sbo_batch_commit(sbo_ctx* ctx, int64_t global_idx);
/* the three steps over the library's communicator (sbo_comm_init): one small all-gather per pick; every rank gets the same picks */
int sbo_safeopt_batch_sharded(sbo_ctx* ctx, int q, sbo_batch_pick* picks, int* n_picked);

/* ---- batch GoOSE acquisition: q distinct safe query points per step (additive; no reference counterpart) ------------
 * The hallucination of the SafeOpt batch above (same noise, same downdate of the objective variance v), over the candidates
 * C = S u T of the local shard: S = SBO_MASK_SAFE of the last sets pass 1, T = the union of the SBO_MASK_TARGET masks of the
 * last GoOSE target stage (Lipschitz mode one per constraint, fantasy mode which = 0, bounds mode the certified members).  The
 * mean does not change; lcb_0(p) = mean_0(p) - beta*sqrt(v(p)) in raw units with the beta of that sets pass.  Pick b, on v
 * conditioned on picks 1..b-1:
 *   S_b = S minus the earlier picks, T_b = T minus the targets earlier explore picks served; S_b empty: no pick;
 *   (safe_idx, safe_lcb) = argmin over S_b of lcb_0, (target_idx, target_lcb) = argmin over T_b (lowest global index on
 *   ties; an empty set gives (-1, +inf));
 *   the rule of test/test_GoOSE.py:158-162: target_idx = -1 or safe_lcb <= target_lcb -> the safe minimum (explore = 0);
 *   else the point of S_b nearest to target_idx in raw coordinates (squared distance as SBO_ARGMIN_DIST, lowest index on
 *   ties; explore = 1), and that target is served.
 * Picks are distinct points of S, so n_picked = min(q, |S|).  Pick 1 is the step's x_new (except after an exact tie of
 * lcb_0 between target points of different constraint masks).  A batch reads the step's state and writes none of it.
 * Every entry point needs a GoOSE target stage (sbo_goose_target after sbo_sets_pass1, or a sharded GoOSE step) since the
 * last model, grid, shard, posterior or set change, and fails with SBO_ERR_INVALID after a SafeOpt pair stage. */
typedef struct sbo_goose_batch_pick {
  int64_t idx;                             /* global index of the pick (a point of S); -1 = no pick */
  int32_t explore, pad;                    /* 0: safe minimum; 1: nearest remaining safe point to target_idx */
  double  safe_lcb;   int64_t safe_idx;    /* min lcb_0 over S_b under the earlier picks (+inf / -1 if empty) */
  double  target_lcb; int64_t target_idx;  /* min lcb_0 over T_b (+inf / -1 if empty) */
  double  dist;                            /* explore: ||x_idx - z_target||_2 in raw units; else 0 */
} sbo_goose_batch_pick;
/* one GPU: at most 5 launches per pick, no host synchronisation between picks, one copy to the host at the end.
 * picks[q] out; *n_picked = min(q, |S|); with S empty picks[0] holds the optima (idx = -1). */
int sbo_goose_batch(sbo_ctx* ctx, int q, sbo_goose_batch_pick* picks, int* n_picked);
/* the same in steps for a grid sharded over ranks; the batch-side state is computed identically on every rank:
 *   sbo_goose_batch_prepare  compact this rank's candidates, v = var_0 (*n_candidates_local = |C| of the shard)
 *   sbo_goose_batch_local    this rank's (safe, target) optima for the next pick, GLOBAL indices (idx / explore apply the
 *                            rule locally; idx = -1 for an explore pick, whose point comes from sbo_goose_batch_nearest)
 *                            -> the caller reduces both (smallest lcb, lowest index) over the ranks
 *   sbo_goose_batch_nearest  explore picks: this rank's point of S_b nearest to the GLOBAL target index, and its SQUARED
 *                            distance (-1 / +inf if S_b is empty here) -> the caller reduces (smallest, lowest index)
 *   sbo_goose_batch_commit   the pick and the target it served (-1: a safe pick), the same on every rank: hallucinate an
 *                            observation at the pick and remove both from S_b / T_b; at most q commits */
int sbo_goose_batch_prepare(sbo_ctx* ctx, int q, int64_t* n_candidates_local);
int sbo_goose_batch_local(sbo_ctx* ctx, sbo_goose_batch_pick* local_optima);
int sbo_goose_batch_nearest(sbo_ctx* ctx, int64_t target_global_idx, int64_t* idx, double* dist2);
int sbo_goose_batch_commit(sbo_ctx* ctx, int64_t pick_global_idx, int64_t served_target_global_idx);
/* the steps over the library's communicator (sbo_comm_init): one small all-gather per pick, a second one for an explore
 * pick; every rank gets the same picks */
int sbo_goose_batch_sharded(sbo_ctx* ctx, int q, sbo_goose_batch_pick* picks, int* n_picked);

/* ---- instrumentation ------------------------------------------------------------------------ */
/* number of kernels this library launched on ctx since the last reset */
int64_t sbo_kernel_launches(sbo_ctx* ctx, int reset);
/* high-water mark (bytes) of the device memory held by the context's work buffers since the last reset */
int64_t sbo_mem_peak(sbo_ctx* ctx, int reset);
/* device time of named phases of the last calls, milliseconds (CUDA events on the ctx stream).
 * phase: 0 model, 1 posterior(crosscov), 2 posterior(solve), 3 sets, 4 pairs, 5 argreduce, 6 pair preparation,
 *        7 FP64 refinement of the split-TF32 fantasy expander, 8 posterior update (sbo_posterior_update) */
int sbo_phase_ms(sbo_ctx* ctx, int phase, double* ms);
/* FP64 refinement of the last pair stage on ctx (fantasy_refine = 2 / 1): the cells the pass was cut into and the FP64 rows
 * V = L^-1 K(X, p) it computed (one cell: one row per distinct candidate and unsafe point of the ambiguous list; more cells
 * compute the inner side's rows once per outer block).  0 / 0 when nothing was refined. */
int sbo_refine_stats(sbo_ctx* ctx, int64_t* cells, int64_t* fp64_rows);
/* tuning / diagnosis options (defaults reproduce the documented behaviour; none changes a result):
 *   "posterior_variant"  1 (default) FP64 tensor cores (DMMA) | 0 FP64 SIMT register tiles
 *   "posterior_tables"   1 (SE kernel only): on meshgrids the cross-covariance kernel multiplies separable SE-ARD factor tables instead of calling
 *                        exp() per entry (same values to ~1e-16 relative; measured slower, 13.5 vs 9.0 ms at C4) | 0 (default)
 *   "posterior_fused"    1 (SE kernel only): meshgrids use separable SE-ARD factor tables; the cross-covariance is generated inside the solve
 *                        kernel's shared-memory stage and never stored (C4: 12 MB of DRAM traffic instead of 33.6 GB, 52.5 ms
 *                        instead of 40.0 ms) | 0 (default): cross-covariance kernel + scratch + solve
 *   "posterior_chunk_mb" size of the cross-covariance tile one posterior chunk keeps between its two kernels in MB (default 1024; 24-96 keeps it L2 resident but measured slower at C4)
 *   "fantasy_variant"    -1 (default) auto | bit 0: 256-column z tiles, bit 1: 8 epilogue warps, bit 2: 2-CTA pairs
 *   "fantasy_gx"         x tile pairs per raster group of the 2-CTA GEMM (0 = default: a quarter of the clusters)
 *   "fantasy_prune"      1 (default): exact pruning of the fantasy expander -- candidates and unsafe points are ordered by the
 *                        Cauchy-Schwarz keys of csrc/pairs.cu (k_key_x / k_key_z) and only tile pairs whose keys can meet
 *                        are evaluated; FP64 counts are unchanged | 0: every pair goes through the GEMM
 *   "prior_mean_zero"    1: zero prior mean for every GP at the next sbo_set_model (GP_Robust.py, StableOpt) | 0 (default) GP_Safe.py:331
 *   "fantasy_refine"     2 (default): the TF32 and TF32X3 fantasy expanders and GoOSE targets settle every pair inside their error bound in FP64
 *                        (the counts are the FP64 counts, at any grid size where the ambiguous pairs fit the list: fewer than 2^31
 *                        per shard) | 1: TF32X3 only | 0: decide on the tensor-core value
 *                        | 3: bounds mode -- no FP64 pass: the counts are the pairs the error bound settles as newly safe (a lower bound
 *                        of the FP64 counts) and sbo_pair_result.n_undecided / undecided_best_* say what is left open (cheaper than
 *                        the FP64 pass, and the mode for shards whose ambiguous pairs do not fit the list)
 *   "fantasy_refine_cap" > 0: initial capacity (pairs) of the ambiguous-pair list instead of the heuristic (test hook)
 *   "fantasy_refine_mb"  device memory of the FP64 refinement (its FP64 rows, their posterior scratch and the cell buckets) in MB:
 *                        0 (default) what cudaMemGetInfo reports free at the start of the pass less 1 GB | > 0 at most this much.
 *                        When the rows of all listed points do not fit, the pass runs cell by cell (blocks of candidates x
 *                        blocks of unsafe points); the counts do not change.  A budget below one row per side: SBO_ERR_NOMEM
 *   "fantasy_f64_variant" 1 (default): FP64 fantasy expander on the FP64 tensor cores (DMMA tiles) | 0: SIMT reference kernel
 *   "pair_cull"          1 (default): exact bounding-box tile culling in the Lipschitz pair kernels | 0 all pairs */
int sbo_set_option(sbo_ctx* ctx, const char* name, int64_t value);
/* ---- hyper-parameter fit:  GP.negative_loglikelihood  (GP_Safe.py:169-192), batched ------
 * NLL_p = y^T K_p^-1 y + log det K_p with K_p = sf2 exp(-1/2 dist) + (sn2 + 1e-8) I for P hyper-parameter vectors at
 * once (a whole differential-evolution population of GP_Safe.py:224 instead of one individual per call).
 * X_norm[n*d] row-major, y[n] (one output column of Y_norm), hyp[P*(d+2)] row p = (1/2 log ell_0..d-1,
 * 1/2 log sf2, 1/2 log sn2) as GP_Safe.py:180-182, nll[P] out; a K_p that is not positive definite gives +inf.
 * Does not touch the model installed by sbo_set_model. */
int sbo_nll_batch(sbo_ctx* ctx, int n, int d, const double* X_norm, const double* y, int P, const double* hyp, double* nll);
/* sbo_nll_batch with K_p = k_p(X, X) + (sn2 + 1e-8) I of the covariance function `kernel` (enum sbo_kernel); sbo_nll_batch is the
 * SBO_KERNEL_SE case. */
int sbo_nll_batch_ex(sbo_ctx* ctx, int kernel, int n, int d, const double* X_norm, const double* y, int P, const double* hyp,
                     double* nll);

/* give device workspaces back to the driver (large grids: the V rows of the fantasy expander are n x count per
 * constraint -- 51 GB per rank at C5).  what = 1: the per-point V rows kept by sbo_posterior(keep_v) (call after
 * sbo_pairs_export_dev; a later fantasy prepare needs a new sbo_posterior); 2: the gathered pair operands
 * (after sbo_pairs_finish_dev); 3: both.  No reference counterpart (the reference never materialises these). */
int sbo_release(sbo_ctx* ctx, int what);

#ifdef __cplusplus
}
#endif
#endif /* SBO_B200_H */
