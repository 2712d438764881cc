// common.cuh -- context, device parameter blocks and helpers shared by the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <type_traits>
#include <vector>
#include "../../include/sbo_b200.h"

#define SBO_EPS_F32 1.1920928955078125e-07   /* jnp.finfo(jnp.float32).eps, GP_Safe.py:229 */
#define SBO_PAIR_OFFSET 1e-8                 /* SafeOpt.py:87 "+1e-8" */

// ---------------------------------------------------------------------------------------------
// device-visible parameter blocks (passed by value)
// ---------------------------------------------------------------------------------------------
struct GridSpec {
  int kind;                 // 1 = implicit meshgrid, 2 = explicit points
  int d;
  long long N;              // global number of points
  long long first, count;   // local shard: contiguous [first, first+count) ...
  int cyc_n, cyc_rank;      // ... or block-cyclic over cyc_n ranks (cyc_n <= 1: contiguous)
  long long cyc_blk;
  long long pts[SBO_MAX_D];
  long long stride[SBO_MAX_D];
  double lo[SBO_MAX_D], hi[SBO_MAX_D], step[SBO_MAX_D];
  const double* explicit_pts;   // [N][d] row-major (global)
};

struct ModelSpec {
  int n, npad, d, G;
  int g0;                   // posterior kernels process GPs g0 .. G-1 (0 except for the constraint-only FP64 rows of the refinement)
  int kernel;               // enum sbo_kernel: the covariance function of every GP of the model
  const double* Xn;         // [npad][d], rows >= n are zero
  const double* alpha;      // [G][npad]
  const double* W;          // [G][npad][npad]  lower-triangular L^-1, zero elsewhere
  double Xmean[SBO_MAX_D], Xstd[SBO_MAX_D];
  double Ymean[SBO_MAX_G], Ystd[SBO_MAX_G], m0[SBO_MAX_G];
  double inv_ell[SBO_MAX_G][SBO_MAX_D];
  double sf2[SBO_MAX_G], sn2[SBO_MAX_G];   // sn2 already includes + eps_f32 (GP_Safe.py:229)
};

// constants of the fantasy expander (constraint GPs only: entry c is GP c+1)
struct FantasyConsts {
  int nc, d, npad;
  int kernel;               // enum sbo_kernel (ModelSpec::kernel)
  double beta;
  double sf2[SBO_MAX_G - 1], sn2[SBO_MAX_G - 1];
  double inv_ell[SBO_MAX_G - 1][SBO_MAX_D];
};

// numpy.linspace coordinate of axis k at index i: lo + i*step (two roundings, no FMA), last = hi.
__device__ __forceinline__ double axis_coord(const GridSpec& g, int k, long long i) {
  if (g.pts[k] > 1 && i == g.pts[k] - 1) return g.hi[k];
  return __dadd_rn(__dmul_rn((double)i, g.step[k]), g.lo[k]);
}
// local shard index -> global grid index
__device__ __host__ __forceinline__ long long shard_global(const GridSpec& g, long long p) {
  if (g.cyc_n > 1) {
    // rotated block-cyclic: in super-block sb (cyc_n consecutive blocks) rank r owns slot (r + rot(sb)) % cyc_n.
    // The rotation keeps a rank from always owning the same slab of a meshgrid whose axis lengths are multiples
    // of block*cyc_n (plain r, r+n, ... put rank 0 on the outer x_1 slab of the 32^4 grid: +20 % unsafe points).
    const long long sb = p / g.cyc_blk, n = g.cyc_n;
    const long long slot = (g.cyc_rank + sb + sb / n + sb / (n * n)) % n;
    return (sb * n + slot) * g.cyc_blk + (p % g.cyc_blk);
  }
  return g.first + p;
}
// raw coordinates of GLOBAL point p
__device__ __forceinline__ void point_coords(const GridSpec& g, long long p, double* x) {
  if (g.kind == 1) {
#pragma unroll
    for (int k = 0; k < SBO_MAX_D; ++k)
      if (k < g.d) x[k] = axis_coord(g, k, (p / g.stride[k]) % g.pts[k]);
  } else {
#pragma unroll
    for (int k = 0; k < SBO_MAX_D; ++k)
      if (k < g.d) x[k] = g.explicit_pts[p * g.d + k];
  }
}

// confidence bounds, rounded like NumPy's  mean -/+ (b*sqrt(var))  (no FMA contraction)   SafeOpt.py:34-45
__device__ __forceinline__ double lcb_of(double mean, double var, double beta) {
  return __dsub_rn(mean, __dmul_rn(beta, sqrt(var)));
}
__device__ __forceinline__ double ucb_of(double mean, double var, double beta) {
  return __dadd_rn(mean, __dmul_rn(beta, sqrt(var)));
}

// ---- packed FP32 (FFMA2 / FMUL2 / FADD2 on sm_100a): two z columns per instruction in the tensor-core epilogue ----
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// ---------------------------------------------------------------------------------------------
// Covariance functions (enum sbo_kernel).  Every kernel site is templated on one of two classes, so an SE model runs the
// code it always ran and Matern 3/2 and 5/2 share one instantiation (their order is a run-time constant).  With the
// scaled squared distance  s = sum_k (x_k - x'_k)^2 / ell_k:
//   value(s, sf2) = k                    SE: sf2 exp(-s/2)      MATERN: sf2 (1 + t + q t^2) exp(-t),  t = sqrt(c s)
//   phi(s, sf2)   = -2 dk/ds              SE: k                  MATERN: c sf2 ((1 - 2q) + q t) exp(-t)
// (Matern 3/2: c = 3, q = 0; 5/2: c = 5, q = 1/3), so that  dk/dx_k = -phi (x_k - x'_k) / ell_k  for every kernel.
// The tensor-core epilogue (fantasy_tc.cu) gets the exponent e from its FP32 records and evaluates k in packed FP32:
//   SE: e = log2 k, k = 2^e.   MATERN: e = -c s (records scaled by rec_scale() = c), k = sf2 P(t) 2^(-t log2 e), t = sqrt(max(-e, 0)).
// ---------------------------------------------------------------------------------------------
struct SE {
  static constexpr bool kIsSE = true;
  __device__ __host__ explicit SE(int) {}
  __device__ __forceinline__ double value(double s, double sf2) const { return sf2 * exp(-0.5 * s); }
  __device__ __forceinline__ double phi(double s, double sf2) const { return sf2 * exp(-0.5 * s); }
  // two columns at once from the packed exponent e; sf2 is already part of e
  __device__ __forceinline__ uint64_t value_f32x2(uint64_t e, uint64_t /*sf2x2*/) const {
    float e0, e1;
    upk2(e, e0, e1);
    return pk2(ex2_approx(e0), ex2_approx(e1));
  }
};
struct MATERN {
  static constexpr bool kIsSE = false;
  double c, q;
  __device__ __host__ explicit MATERN(int kernel)
      : c(kernel == SBO_KERNEL_MATERN32 ? 3.0 : 5.0), q(kernel == SBO_KERNEL_MATERN32 ? 0.0 : 1.0 / 3.0) {}
  __device__ __forceinline__ double value(double s, double sf2) const {
    const double t = sqrt(c * s);
    return sf2 * fma(fma(q, t, 1.0), t, 1.0) * exp(-t);
  }
  __device__ __forceinline__ double phi(double s, double sf2) const {
    const double t = sqrt(c * s);
    return c * sf2 * fma(q, t, 1.0 - 2.0 * q) * exp(-t);
  }
  // e = -c s of two columns (clamped at 0: the expanded square can round below it); sf2x2 = (sf2, sf2)
  __device__ __forceinline__ uint64_t value_f32x2(uint64_t e, uint64_t sf2x2) const {
    float e0, e1;
    upk2(e, e0, e1);
    const uint64_t t = pk2(sqrt_approx(fmaxf(-e0, 0.f)), sqrt_approx(fmaxf(-e1, 0.f)));
    const float nl = -1.4426950408889634f, qf = (float)q;
    float y0, y1;
    upk2(mul2(t, pk2(nl, nl)), y0, y1);
    const uint64_t ex = pk2(ex2_approx(y0), ex2_approx(y1));
    const uint64_t P = fma2(fma2(pk2(qf, qf), t, pk2(1.f, 1.f)), t, pk2(1.f, 1.f));
    return mul2(mul2(P, sf2x2), ex);
  }
};
// scale of the squared-distance terms of the FP32 records: SE log2(e)/2 (e = log2 k), MATERN c (e = -c s)
static inline double kernel_rec_scale(int kernel) {
  return kernel == SBO_KERNEL_SE ? 0.5 * 1.4426950408889634 : (kernel == SBO_KERNEL_MATERN32 ? 3.0 : 5.0);
}
static inline bool kernel_valid(int kernel) {
  return kernel == SBO_KERNEL_SE || kernel == SBO_KERNEL_MATERN32 || kernel == SBO_KERNEL_MATERN52;
}
// Host-side compile-time dispatch: each helper calls f with a value that names one template argument and returns what
// f returns, so nested calls select one kernel instantiation and can hand back an SBO status.
// f(SE{}) or f(MATERN{kernel}) -- f launches the instantiation of its kernel class
template <class F>
static inline auto with_kernel(int kernel, F&& f) {
  if (kernel == SBO_KERNEL_SE) return f(SE(kernel));
  return f(MATERN(kernel));
}
// f(std::integral_constant<int, v>{}) for v in [LO, HI]; any other v takes HI (callers validate v)
template <int LO, int HI, class F>
static inline auto with_int(int v, F&& f) {
  if constexpr (LO < HI) {
    if (v != LO) return with_int<LO + 1, HI>(v, f);
  }
  return f(std::integral_constant<int, LO>{});
}
// f(std::true_type{}) or f(std::false_type{})
template <class F>
static inline auto with_flag(bool b, F&& f) {
  if (b) return f(std::true_type{});
  return f(std::false_type{});
}
// keep_v of the posterior whose V rows the fantasy pair test of this precision reads
static inline int keep_v_of(int precision) {
  return precision == SBO_PREC_FP64 ? 1 : (precision == SBO_PREC_TF32 ? 2 : 3);
}

// (value, index) pairs with lowest-index tie-break
struct ArgVal { double v; long long i; };
__device__ __forceinline__ ArgVal argmin2(ArgVal a, ArgVal b) {
  return (b.v < a.v || (b.v == a.v && b.i < a.i)) ? b : a;
}
__device__ __forceinline__ ArgVal argmax2(ArgVal a, ArgVal b) {
  return (b.v > a.v || (b.v == a.v && b.i < a.i)) ? b : a;
}
__device__ __forceinline__ ArgVal shfl_xor_argval(ArgVal a, int m) {
  ArgVal r;
  r.v = __shfl_xor_sync(0xffffffffu, a.v, m);
  r.i = __shfl_xor_sync(0xffffffffu, a.i, m);
  return r;
}
#define SBO_IDX_NONE 0x7fffffffffffffffLL

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

// state of the staged pair driver (pairs.cu)
struct PairStage {
  bool prepared = false, imported = false, counted = false, sorted = false;   // sorted: fantasy operands in key order (exact pruning)
  bool exportable = false;   // prepared, and a fantasy stage's V rows (what sbo_pairs_export reads) not released since
  int mode = 0, precision = 0, row_doubles = 0, count_scale = 1;
  double beta = 0.0;
  double L[SBO_MAX_G] = {0, 0, 0, 0, 0, 0, 0, 0};   // L[c] for constraint c+1
  long long nx_local = 0, nz_local = 0, nz_full = 0, nx_total = 0, pairs_evaluated = 0;   // nz_local <= nz_full when pruned
  // sharded runs: candidates per rank (prefix sums), this rank; canon: payloads re-ordered to grid order at import;
  // nz_global >= 0: the Lipschitz expander pairs this rank's candidate tiles with ALL unsafe points (gz_* buffers)
  int seg_n = 1, seg_rank = 0;
  long long seg_off[65] = {0};
  bool canon = false;
  long long nz_global = -1;
  bool bounds = false;                               // fantasy_refine = 3: counts are settled lower bounds, amb_rows the undecided pairs
  long long n_ambiguous = 0, n_refined_safe = 0;     // split-TF32 refinement statistics of the last run
};

// state of a batch SafeOpt or GoOSE acquisition (batch.cu)
struct BatchRec {                 // device record of one pick: raw objective variances, GLOBAL indices (-1 = empty)
  long long idx;
  int from_exp, pad;
  double vmin; long long imin;
  double vexp; long long iexp;
};
struct BatchStage {
  bool prepared = false;
  bool goose = false;             // prepared for the GoOSE rule (C = S u T) instead of SafeOpt's (C = M u E)
  int q = 0, b = 0;               // picks asked for / observations hallucinated so far
  long long nc = 0;               // local candidates |C|
  int nparts = 0;                 // block partials of the candidate kernel
};

struct sbo_comm;   // comm.cu: NCCL communicator + gathered buffers

struct sbo_ctx {
  int device = 0;
  sbo_comm* comm = nullptr;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  std::string err;
  int64_t launches = 0;
  int64_t mem_now = 0, mem_peak = 0;   // device bytes held by the context's work buffers (sbo_ensure), and their high-water mark

  // model
  bool have_model = false;
  ModelSpec ms{};
  DevBuf Xn, Yn, alpha, W, Kmat, info;
  // grid
  bool have_grid = false;
  GridSpec gs{};
  DevBuf pts;
  // posterior (local shard)
  int post_g0 = 0;           // first GP the posterior kernels process (posterior_vrows_dev: constraints only)
  bool have_post = false, have_grad = false;   // have_grad: the last posterior accumulated the Lipschitz constants
  DevBuf mean, var, kx, lmax, tabs;     // tabs: separable SE-ARD factor tables of the meshgrid (posterior.cu)
  int keep_v = 0;            // 0 none, 1 fp64, 2 fp32
  DevBuf vall;               // [(G-1)][count][npad] rows of V for the constraints
  // the last posterior_run as sbo_posterior_update sees it: valid while the model changed only through sbo_append_sample
  // (model n and npad, the flags it ran with)
  struct { bool valid = false, with_grad = false; int n = 0, npad = 0, keep_v = 0; } up;
  // sets
  bool have_sets = false, have_sets2 = false;
  bool have_exp = false;     // the last pair stage was a SafeOpt expander on the current sets (m_exp valid; batch.cu needs it)
  bool have_tgt = false;     // the same for a GoOSE target stage (m_tgt valid; the GoOSE batch needs it)
  double beta = 0.0;
  DevBuf m_safe, m_unsafe, m_min, m_user, m_exp, m_tgt;
  DevBuf partials, result;
  // compaction / pair workspaces
  DevBuf scan_a, scan_b, xs_idx, zs_idx, xs_pay, zs_pay, hits, counts, pairctr;
  DevBuf imp_rows;
  DevBuf vx, vz, aux_x, aux_z;
  DevBuf pp_x, pp_m, pp_v, pp_k, pp_g;   // scratch of the arbitrary-point posterior calls
  DevBuf tc_stats;                        // maxima behind the absolute error terms of the refining epilogue
  DevBuf tc_row, tc_col, tc_err;          // FP32 row/column records of the tcgen05 fantasy kernel
  DevBuf nll_K, nll_in;                   // batched NLL (hyper-parameter fit): P x npad x npad factors, inputs/outputs
  DevBuf tile_bb;                         // bounding boxes of the staged tiles (Lipschitz pair kernels)
  DevBuf exp_rows, exp_v;                 // single-GPU export buffers of the staged pair driver
  DevBuf key_x, key_z, perm_x, perm_z, sort_ws, tile_keys, item_mask, item_list;   // exact pruning of the fantasy expander
  DevBuf amb_list, amb_ctr, amb_mask, amb_xd, amb_zd, amb_rx, amb_rz, amb_pts, amb_vx, amb_vz, amb_rows, m_und;   // FP64 refinement of the split-TF32 expander
  DevBuf amb_cell, amb_hist;              // cell-wise refinement: the ambiguous list bucketed by cell, per-cell counters
  DevBuf amb_tgt;                         // GoOSE target refinement: the listed pairs whose z is not yet in the target set
  int64_t refine_cells = 0, refine_rows = 0;   // last pair stage: cells of the FP64 refinement and FP64 rows computed (sbo_refine_stats)
  DevBuf st_score, st_mask;               // StableOpt: per-x_c worst-case score and robust-safe bitmask
  DevBuf gz_mask, gz_idx, gz_pay;         // all-gathered unsafe set of a sharded Lipschitz expander
  PairStage ps;
  BatchStage bt;
  DevBuf bt_mask, bt_idx, bt_flag, bt_v, bt_w, bt_part, bt_pick;   // batch: C = M u E (S u T), membership bits, v[C], w[q][C], partials, pick side
  // timing: event pairs are recorded without host syncs and summed per phase by ev_collect()
  struct EvPair { cudaEvent_t a, b; int phase; };
  std::vector<EvPair> evlog;
  std::vector<cudaEvent_t> evpool;
  double phase_ms[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  // options
  int64_t opt_posterior_variant = 1;  // 0: FP64 SIMT register tiles, 1: FP64 tensor cores (DMMA m8n8k4)
  int64_t opt_fantasy_prune = 1;      // 1 (default): exact key-ordered tile pruning of the fantasy expander (pairs.cu); 0: every pair
  long long n_unsafe_local = 0;
  long long n_safe_local = 0;         // |S| of the local shard after the last sets pass 1 (the GoOSE batch's pick count)
  int64_t opt_fantasy_variant = -1;  // -1 auto; bit 0: BN=256 (2 TMEM slots) instead of 128 (4 slots); bit 1: 8 epilogue warps;
                                     // bit 2: 2-CTA pairs (cta_group::2, 256x256 tile pairs)
  int64_t opt_posterior_fused = 0;    // 1: meshgrid: separable factor tables + fused solve, no cross-covariance scratch (12 MB instead of 33.6 GB
                                      // of DRAM traffic at C4, but 52.5 vs 40.0 ms: the table loads stall the DMMA loop) | 0 (default): two kernels + scratch
  int64_t opt_posterior_tables = 0;   // 1: meshgrid cross-covariance values from the separable factor tables instead of exp() (measured slower:
                                      // 13.5 vs 9.0 ms at C4 -- the kernel is bound by its Kx stores and address stream, not by exp)
  int64_t opt_posterior_chunk_mb = 0; // Kx scratch per chunk in MB (0 = default 1024; never less than one wave of the solve, posterior.cu chunk_points)
  int64_t opt_prior_mean_zero = 0;    // 1: zero prior mean for every GP (GP_Robust.py:322-323, StableOpt); 0: GP_Safe.py:331-332
  int64_t opt_fantasy_f64_variant = 1; // FP64 fantasy expander: 1 (default) tensor cores (DMMA 128x64 tiles) | 0 SIMT reference kernel
  int64_t opt_fantasy_refine = 2;     // tensor-core fantasy expander: pairs the FP32/TF32 error bound cannot settle are re-evaluated in FP64 (exact
                                      // counts): 2 (default) TF32 and TF32X3, 1 TF32X3 only, 0 off (decide on the tensor-core value)
  int64_t opt_fantasy_refine_cap = 0; // > 0: initial capacity of the ambiguous-pair list (tests force the overflow / re-run path with it)
  int64_t opt_fantasy_refine_mb = 0;  // device memory of the FP64 refinement pass in MB: 0 (default) what is free, > 0 at most this
  int64_t opt_pair_cull = 1;         // Lipschitz pair kernels: exact bounding-box culling of staged tiles
  int64_t opt_fantasy_gx = 0;        // 2-CTA kernel: x tile pairs per raster group (0 = default)
};

// What a call did to the pipeline  model -> posterior -> sets pass 1 (-> pass 2) -> pair stage -> batch.  stage_changed()
// (capi.cu) decides what that leaves valid; no other code writes have_post, have_grad, have_sets(2), have_exp, have_tgt,
// keep_v, up.valid, ps.prepared / imported / exportable or bt.prepared.
enum class Change {
  MODEL,            // sbo_set_model(_ex) starts replacing the model
  APPEND,           // sbo_append_sample starts growing it: the last posterior can still be updated
  GRID,             // sbo_set_grid / _points / _shard / _shard_cyclic
  POSTERIOR,        // a posterior run starts overwriting mean, var and the kept V rows
  POSTERIOR_DONE,   // a posterior run or update completed with the flags in ctx->up
  SETS1, SETS2,     // a sets pass completed
  PAIRS,            // sbo_pairs_prepare starts a new pair stage
  PAIRS_PREPARED, PAIRS_IMPORTED,
  EXPANDER, TARGET, // sbo_pairs_finish_dev completed the SafeOpt expander / GoOSE target masks
  BATCH,            // a batch starts its prepare, or ran whole: the staged batch calls need a new prepare
  BATCH_PREPARED,
  RELEASE_V,        // sbo_release(1)
  RELEASE_PAIRS,    // sbo_release(2)
};
void stage_changed(sbo_ctx* ctx, Change c);

extern thread_local std::string g_sbo_last_error;

int sbo_fail(sbo_ctx* ctx, int code, const std::string& msg);
int sbo_ensure(sbo_ctx* ctx, DevBuf& b, size_t bytes);
int sbo_ensure_exact(sbo_ctx* ctx, DevBuf& b, size_t bytes);   // as sbo_ensure, without the 1/8 head-room
void sbo_free(sbo_ctx* ctx, DevBuf& b);                         // give a work buffer back to the driver

#define SBO_CUDA(call)                                                                         \
  do {                                                                                         \
    cudaError_t e__ = (call);                                                                  \
    if (e__ != cudaSuccess)                                                                    \
      return sbo_fail(ctx, SBO_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
  } while (0)
#define SBO_TRY(call)            \
  do {                           \
    int r__ = (call);            \
    if (r__ != SBO_OK) return r__; \
  } while (0)
#define SBO_REQUIRE(cond, msg) \
  do {                         \
    if (!(cond)) return sbo_fail(ctx, SBO_ERR_INVALID, msg); \
  } while (0)
#define SBO_LAUNCH_CHECK()                                                                      \
  do {                                                                                          \
    ctx->launches++;                                                                            \
    cudaError_t e__ = cudaGetLastError();                                                       \
    if (e__ != cudaSuccess)                                                                     \
      return sbo_fail(ctx, SBO_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(e__) + \
                                             " at " + __FILE__ + ":" + std::to_string(__LINE__)); \
  } while (0)

// phase ids: 0 model, 1 posterior cross-covariance, 2 posterior solve, 3 sets, 4 pairs, 5 arg-reduce, 6 pair prep,
// 7 FP64 refinement, 8 posterior update
void ev_begin(sbo_ctx* ctx, int phase);   // record a start event on the ctx stream
void ev_end(sbo_ctx* ctx);                // record the matching stop event
void ev_reset(sbo_ctx* ctx, int phase);   // zero a phase accumulator
void ev_collect(sbo_ctx* ctx);            // (after a stream sync) add all logged pairs to phase_ms

static inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }

// implemented across the .cu files
int model_upload(sbo_ctx* ctx, int kernel, int n, int d, int G, const double* X_norm, const double* Y_norm,
                 const double* X_mean, const double* X_std, const double* Y_mean, const double* Y_std,
                 const double* hyp);
int model_append(sbo_ctx* ctx, const double* x_norm_new, const double* y_norm_new);
int ball_mask(sbo_ctx* ctx, int mask_kind, const double* x0, double r);
int stable_minmax(sbo_ctx* ctx, int n_controlled, int fun_kind, double beta, int64_t* xc_idx, double* value, int64_t* n_robust_safe, double* score_host);
int nll_batch(sbo_ctx* ctx, int kernel, int n, int d, const double* X_norm, const double* y, int P, const double* hyp, double* nll);
int posterior_run(sbo_ctx* ctx, int with_grad, int keep_v);
int posterior_update(sbo_ctx* ctx, sbo_update_info* info);
int posterior_vrows_dev(sbo_ctx* ctx, long long m, const double* pts_dev, double* vout);
void posterior_vrows_scratch(const sbo_ctx* ctx, long long m, size_t* mv_bytes, size_t* k_bytes);
int posterior_points(sbo_ctx* ctx, int64_t m, const double* x, double* mean, double* var);
int posterior_point_grad(sbo_ctx* ctx, int gp, int64_t m, const double* x, double* grad);
int sets_pass1(sbo_ctx* ctx, double beta, int rule, int strict, sbo_sets_result* out);
int sets_pass2(sbo_ctx* ctx, double min_ucb0, sbo_sets_result* out);
int argreduce_run(sbo_ctx* ctx, int kind, const uint32_t* mask_dev, const double* target_host, int64_t* idx, double* value);
int compact_mask(sbo_ctx* ctx, const uint32_t* mask_dev, long long count, DevBuf& out_idx, long long* n_out);
int pairs_lipschitz(sbo_ctx* ctx, bool goose, double beta, const double* L, sbo_pair_result* out);
int pairs_prepare(sbo_ctx* ctx, int mode, int precision, double beta, const double* L, sbo_pairs_info* info);
int pairs_export(sbo_ctx* ctx, void* rows_dev, void* vrows_dev);
int pairs_import(sbo_ctx* ctx, long long n_total, const void* rows_dev, const void* vrows_dev);
int pairs_run(sbo_ctx* ctx, int goose, void* result_dev);
int pairs_set_segments(sbo_ctx* ctx, int nranks, int rank, const int64_t* n_per_rank);
int pairs_goose_localize(sbo_ctx* ctx, const void* hits_global, void* hits_local);
int pairs_set_global_unsafe(sbo_ctx* ctx, const void* gathered_words_dev, long long words_per_rank, int nranks);
int pairs_finish(sbo_ctx* ctx, int goose, long long offset, const void* result_dev, sbo_pair_result* out, int32_t* counts_host);
int pairs_fantasy(sbo_ctx* ctx, int precision, double beta, sbo_pair_result* out, int32_t* counts_host);
int pairs_goose_fantasy(sbo_ctx* ctx, int precision, double beta, sbo_pair_result* out);
int batch_prepare(sbo_ctx* ctx, int q, long long* n_candidates);
int batch_local(sbo_ctx* ctx, BatchRec* out);
int batch_commit(sbo_ctx* ctx, long long global_idx);
void batch_pick_of(const BatchRec& r, sbo_batch_pick* out);
int goose_batch_prepare(sbo_ctx* ctx, int q, long long* n_candidates);
int goose_batch_local(sbo_ctx* ctx, sbo_goose_batch_pick* out);
int goose_batch_nearest(sbo_ctx* ctx, long long target, long long* idx, double* dist2);
int goose_batch_commit(sbo_ctx* ctx, long long pick, long long served_target);
uint32_t* mask_ptr(sbo_ctx* ctx, int mask_kind, int which);
long long mask_words(const sbo_ctx* ctx);
