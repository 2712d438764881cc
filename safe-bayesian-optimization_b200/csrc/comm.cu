// comm.cu -- library-owned communicator and whole sharded acquisition steps behind the C ABI (SURVEY.md section 8b
// "sbo_comm_init(ctx, rank, nranks, ncclUniqueId)", 8e).  One process per GPU, one context per process; the grid is
// sharded with sbo_set_shard_cyclic.  NCCL is resolved at run time (dlopen "libnccl.so.2"), so the library keeps
// loading on a machine without NCCL or a GPU driver and a host that is not PyTorch (the reference is JAX/NumPy) can
// shard the step.  Collectives, all issued on the context's stream (ordered with its kernels, no host syncs between):
//   all-gather   one small record per stage (local optima as (value, global index), counts, Lipschitz constants);
//                reduced on the host: best value, lowest index on ties -> every rank gets the same answer
//   broadcast    (grouped, one per rank) candidate rows / V rows written straight into the gathered buffer
//   all-gather   unsafe bitmask (Lipschitz SafeOpt expander: N/8 bytes in total)
//   all-reduce   per-candidate hit flags (max) / newly-safe counts (sum); none for the fantasy GoOSE target, whose
//                verdict on an unsafe point is local (every rank pairs all candidates with its own unsafe points)
// Decision rules: test/test_SafeOpt.py:144-158 and test/test_GoOSE.py:151-162 of the reference.
#include "common.cuh"
#include <dlfcn.h>
#include <math.h>
#include <string.h>

// ---- the slice of nccl.h this file needs (NCCL 2.x ABI) ---------------------------------------------------------
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclInt8 = 0, ncclUint8 = 1, ncclInt32 = 2, ncclFloat64 = 8 };
enum { ncclSum = 0, ncclMax = 2 };

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

static int nccl_load(sbo_ctx* ctx) {
  if (g_nccl.lib) return SBO_OK;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);     // reuses the copy a host framework already loaded
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return sbo_fail(ctx, SBO_ERR_INVALID, std::string("NCCL is not available: ") + dlerror());
#define SYM(field, name)                                                                                     \
  *(void**)(&g_nccl.field) = dlsym(h, name);                                                                 \
  if (!g_nccl.field) return sbo_fail(ctx, SBO_ERR_INVALID, std::string("NCCL symbol missing: ") + name)
  SYM(GetUniqueId, "ncclGetUniqueId"); SYM(CommInitRank, "ncclCommInitRank"); SYM(CommDestroy, "ncclCommDestroy");
  SYM(AllReduce, "ncclAllReduce"); SYM(AllGather, "ncclAllGather"); SYM(Broadcast, "ncclBroadcast");
  SYM(GroupStart, "ncclGroupStart"); SYM(GroupEnd, "ncclGroupEnd"); SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
  g_nccl.lib = h;
  return SBO_OK;
}

#define SBO_NCCL(call)                                                                                     \
  do {                                                                                                     \
    ncclResult_t r__ = (call);                                                                             \
    if (r__ != 0) return sbo_fail(ctx, SBO_ERR_CUDA, std::string(#call) + ": " + g_nccl.GetErrorString(r__)); \
  } while (0)

struct sbo_comm {
  ncclComm_t comm = nullptr;
  int rank = 0, nranks = 1;
  DevBuf small, rows, vrows, result, masks;     // gathered records / candidate rows / V rows / results / unsafe masks
};

static ncclComm_t NC(sbo_ctx* ctx) { return ctx->comm->comm; }

// all-gather `n` doubles per rank through the device, reduced by the caller on the host: out[r*n + k]
static int gather_record(sbo_ctx* ctx, const double* mine, int n, std::vector<double>& out) {
  sbo_comm* cm = ctx->comm;
  SBO_TRY(sbo_ensure(ctx, cm->small, sizeof(double) * (size_t)n * (cm->nranks + 1)));
  double* send = (double*)cm->small.p;
  double* recv = send + n;
  SBO_CUDA(cudaMemcpyAsync(send, mine, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
  SBO_NCCL(g_nccl.AllGather(send, recv, (size_t)n, ncclFloat64, NC(ctx), ctx->stream));
  out.resize((size_t)n * cm->nranks);
  SBO_CUDA(cudaMemcpyAsync(out.data(), recv, sizeof(double) * out.size(), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}

// best (value, index) over the ranks of field pair (k, k+1) of the gathered records: lowest index on ties, -1 = empty
static void reduce_arg(const std::vector<double>& g, int n, int nranks, int k, bool maximize, double* v, int64_t* i) {
  double bv = maximize ? -INFINITY : INFINITY;
  int64_t bi = -1;
  for (int r = 0; r < nranks; ++r) {
    const double val = g[(size_t)r * n + k];
    const int64_t idx = (int64_t)g[(size_t)r * n + k + 1];          // indices < 2^53 are exact in a double
    if (idx < 0) continue;
    if (bi < 0 || (maximize ? val > bv : val < bv) || (val == bv && idx < bi)) { bv = val; bi = idx; }
  }
  *v = bv; *i = bi;
}

// the pair stage of one step on the sharded grid; `pr` gets GLOBAL optima (identical on every rank)
// s2 (optional): this rank's pass-2 result (minimiser); its reduction rides on the first gather of the pair stage and is
// written to sets_out, so that a step needs three small all-gathers instead of five
static int sharded_pairs(sbo_ctx* ctx, int mode, int precision, bool goose, double beta, const double* L, sbo_pair_result* pr,
                         const sbo_sets_result* s2 = nullptr, sbo_sets_result* sets_out = nullptr) {
  sbo_comm* cm = ctx->comm;
  const int R = cm->nranks, rank = cm->rank;
  const int nc = ctx->ms.G - 1;
  const bool fantasy = mode == SBO_MODE_FANTASY;
  sbo_pairs_info info;
  SBO_TRY(pairs_prepare(ctx, mode, precision, beta, L, &info));
  // (1) candidate counts of every rank
  std::vector<double> g;
  double mine1[6] = {(double)info.n_x_local, (double)info.n_z_local, (double)mask_words(ctx),
                     s2 ? s2->minimizer_var : 0.0, s2 ? (double)s2->minimizer_idx : -1.0, s2 ? (double)s2->n_min : 0.0};
  SBO_TRY(gather_record(ctx, mine1, 6, g));
  std::vector<int64_t> n_all(R);
  int64_t n_total = 0, offset = 0, nz_total = 0;
  long long wpr = 0;
  for (int r = 0; r < R; ++r) {
    n_all[r] = (int64_t)g[6 * r];
    if (r < rank) offset += n_all[r];
    n_total += n_all[r];
    nz_total += (int64_t)g[6 * r + 1];
    wpr = wpr > (long long)g[6 * r + 2] ? wpr : (long long)g[6 * r + 2];
  }
  if (s2 && sets_out) {
    reduce_arg(g, 6, R, 3, true, &sets_out->minimizer_var, &sets_out->minimizer_idx);
    sets_out->n_min = 0;
    for (int r = 0; r < R; ++r) sets_out->n_min += (int64_t)g[6 * r + 5];
  }
  // (2) export into the gathered buffers, complete them with one grouped broadcast per rank
  const size_t row_b = sizeof(double) * (size_t)info.row_doubles, v_b = (size_t)info.vrow_bytes;
  SBO_TRY(sbo_ensure(ctx, cm->rows, row_b * (size_t)(n_total > 0 ? n_total : 1)));
  if (v_b) SBO_TRY(sbo_ensure(ctx, cm->vrows, v_b * (size_t)(n_total > 0 ? n_total : 1)));
  char* rows = (char*)cm->rows.p;
  char* vrows = v_b ? (char*)cm->vrows.p : nullptr;
  SBO_TRY(pairs_export(ctx, rows + row_b * offset, vrows ? vrows + v_b * offset : nullptr));
  const bool big = v_b * (size_t)n_total > ((size_t)4 << 30);
  if (big) SBO_TRY(sbo_release(ctx, 1));                       // per-point V rows are not needed after the export
  SBO_NCCL(g_nccl.GroupStart());
  {
    int64_t off = 0;
    for (int r = 0; r < R; ++r) {
      if (n_all[r]) {
        SBO_NCCL(g_nccl.Broadcast(rows + row_b * off, rows + row_b * off, row_b * (size_t)n_all[r], ncclInt8, r, NC(ctx), ctx->stream));
        if (vrows) SBO_NCCL(g_nccl.Broadcast(vrows + v_b * off, vrows + v_b * off, v_b * (size_t)n_all[r], ncclInt8, r, NC(ctx), ctx->stream));
      }
      off += n_all[r];
    }
  }
  SBO_NCCL(g_nccl.GroupEnd());
  // (3) reference-exact mode: grid order of the gathered candidates; SafeOpt expander split by candidates
  if (!fantasy && R > 1) {
    SBO_TRY(pairs_set_segments(ctx, R, rank, n_all.data()));
    {   // SafeOpt expander: split by candidates; GoOSE target: split by (grid-ordered) unsafe tiles -- both over ALL unsafe points
      SBO_TRY(sbo_ensure(ctx, cm->masks, sizeof(uint32_t) * (size_t)wpr * (R + 1)));
      uint32_t* loc = (uint32_t*)cm->masks.p;
      uint32_t* all = loc + wpr;
      SBO_TRY(sbo_mask_export_dev(ctx, SBO_MASK_UNSAFE, 0, loc, wpr));
      SBO_NCCL(g_nccl.AllGather(loc, all, (size_t)wpr, ncclInt32, NC(ctx), ctx->stream));
      SBO_TRY(pairs_set_global_unsafe(ctx, all, wpr, R));
    }
  }
  SBO_TRY(pairs_import(ctx, n_total, rows, vrows));
  if (big) { SBO_CUDA(cudaStreamSynchronize(ctx->stream)); cudaFree(cm->vrows.p); ctx->mem_now -= (int64_t)cm->vrows.cap; cm->vrows.p = nullptr; cm->vrows.cap = 0; }
  // (4) run on the local shard, combine the per-candidate results
  const long long nzg = ctx->ps.nz_global;                     // >= 0: the pair stage runs over the all-gathered unsafe set
  const bool goose_global = goose && nzg >= 0;
  const size_t res_b = fantasy ? (goose ? sizeof(uint32_t) * (size_t)cdiv(info.n_z_local, 32) : sizeof(int) * (size_t)n_total)
                               : (size_t)nc * (size_t)(goose ? (goose_global ? nzg : info.n_z_local) : n_total);
  SBO_TRY(sbo_ensure(ctx, cm->result, (res_b ? res_b : 16) + (goose_global ? (size_t)nc * info.n_z_local + 16 : 0)));
  SBO_TRY(pairs_run(ctx, goose ? 1 : 0, cm->result.p));
  if (!goose && n_total > 0) {
    if (fantasy) {
      SBO_NCCL(g_nccl.AllReduce(cm->result.p, cm->result.p, (size_t)n_total, ncclInt32, ncclSum, NC(ctx), ctx->stream));
      if (ctx->ps.bounds)    // bounds mode: the per-candidate undecided-pair counts are combined like the settled counts
        SBO_NCCL(g_nccl.AllReduce(ctx->amb_rows.p, ctx->amb_rows.p, (size_t)n_total, ncclInt32, ncclSum, NC(ctx), ctx->stream));
    }
    else SBO_NCCL(g_nccl.AllReduce(cm->result.p, cm->result.p, (size_t)nc * n_total, ncclUint8, ncclMax, NC(ctx), ctx->stream));
  }
  const void* res_ptr = cm->result.p;
  if (goose_global && nzg > 0 && n_total > 0) {
    SBO_NCCL(g_nccl.AllReduce(cm->result.p, cm->result.p, (size_t)nc * nzg, ncclUint8, ncclMax, NC(ctx), ctx->stream));
    unsigned char* local = (unsigned char*)cm->result.p + (((size_t)nc * nzg + 15) & ~(size_t)15);
    SBO_TRY(pairs_goose_localize(ctx, cm->result.p, local));
    res_ptr = local;
  }
  sbo_pair_result loc;
  SBO_TRY(pairs_finish(ctx, goose ? 1 : 0, goose ? 0 : offset, res_ptr, &loc, nullptr));
  // (5) global optima: per constraint (value, index), then the first best over the constraints (SafeOpt.py:120-122)
  const int nmask = fantasy ? 1 : nc;
  const int nrec = 2 * SBO_MAX_G + 8;
  double mine2[2 * SBO_MAX_G + 8];
  for (int c = 0; c < SBO_MAX_G; ++c) { mine2[2 * c] = loc.per_value[c]; mine2[2 * c + 1] = (double)loc.per_idx[c]; }
  mine2[2 * SBO_MAX_G] = (double)loc.n_hit; mine2[2 * SBO_MAX_G + 1] = (double)loc.pairs_evaluated;
  mine2[2 * SBO_MAX_G + 2] = (double)loc.n_ambiguous; mine2[2 * SBO_MAX_G + 3] = (double)loc.n_refined_safe;
  mine2[2 * SBO_MAX_G + 4] = loc.undecided_best_value; mine2[2 * SBO_MAX_G + 5] = (double)loc.undecided_best_idx;
  mine2[2 * SBO_MAX_G + 6] = (double)loc.n_undecided; mine2[2 * SBO_MAX_G + 7] = 0.0;
  SBO_TRY(gather_record(ctx, mine2, nrec, g));
  memset(pr, 0, sizeof(*pr));
  pr->best_idx = -1; pr->best_value = goose ? INFINITY : -INFINITY;
  for (int c = 0; c < SBO_MAX_G; ++c) { pr->per_idx[c] = -1; pr->per_value[c] = goose ? INFINITY : -INFINITY; }
  for (int c = 0; c < nmask; ++c) {
    reduce_arg(g, nrec, R, 2 * c, !goose, &pr->per_value[c], &pr->per_idx[c]);
    if (pr->per_idx[c] >= 0 && (pr->best_idx < 0 || (goose ? pr->per_value[c] < pr->best_value : pr->per_value[c] > pr->best_value))) {
      pr->best_idx = pr->per_idx[c]; pr->best_value = pr->per_value[c];
    }
  }
  for (int r = 0; r < R; ++r) {
    pr->n_hit += (int64_t)g[(size_t)r * nrec + 2 * SBO_MAX_G]; pr->pairs_evaluated += (int64_t)g[(size_t)r * nrec + 2 * SBO_MAX_G + 1];
    pr->n_ambiguous += (int64_t)g[(size_t)r * nrec + 2 * SBO_MAX_G + 2]; pr->n_refined_safe += (int64_t)g[(size_t)r * nrec + 2 * SBO_MAX_G + 3];
  }
  reduce_arg(g, nrec, R, 2 * SBO_MAX_G + 4, !goose, &pr->undecided_best_value, &pr->undecided_best_idx);   // GoOSE: min lcb_0
  for (int r = 0; r < R; ++r) pr->n_undecided += (int64_t)g[(size_t)r * nrec + 2 * SBO_MAX_G + 6];
  pr->n_x = n_total; pr->n_z = nz_total; pr->pairs_algorithmic = n_total * nz_total * nc;
  if (big) SBO_TRY(sbo_release(ctx, 2));
  return SBO_OK;
}

// posterior + both set passes on the sharded grid; fills the set part of `out`
static int sharded_sets(sbo_ctx* ctx, double beta, int unsafe_rule, int with_grad, int keep_v, sbo_sets_result* s2_local, sbo_step_result* out) {
  sbo_comm* cm = ctx->comm;
  const int R = cm->nranks, G = ctx->ms.G;
  SBO_TRY(posterior_run(ctx, with_grad, keep_v));
  sbo_sets_result s1;
  SBO_TRY(sets_pass1(ctx, beta, unsafe_rule, 0, &s1));
  const int n1 = 6 + SBO_MAX_G;
  double mine[6 + SBO_MAX_G] = {s1.min_ucb0, (double)s1.min_ucb0_idx, s1.min_lcb0, (double)s1.min_lcb0_idx, (double)s1.n_safe, (double)s1.n_unsafe};
  if (with_grad) {
    double Lh[SBO_MAX_G] = {0};
    SBO_CUDA(cudaMemcpyAsync(Lh, ctx->lmax.p, sizeof(double) * G, cudaMemcpyDeviceToHost, ctx->stream));
    SBO_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < G; ++i) mine[6 + i] = Lh[i];
  }
  std::vector<double> g;
  SBO_TRY(gather_record(ctx, mine, n1, g));
  reduce_arg(g, n1, R, 0, false, &out->sets.min_ucb0, &out->sets.min_ucb0_idx);
  reduce_arg(g, n1, R, 2, false, &out->sets.min_lcb0, &out->sets.min_lcb0_idx);
  out->sets.n_safe = out->sets.n_unsafe = out->sets.n_min = 0;
  for (int i = 0; i < SBO_MAX_G; ++i) out->L[i] = 0.0;
  for (int r = 0; r < R; ++r) {
    out->sets.n_safe += (int64_t)g[(size_t)r * n1 + 4];
    out->sets.n_unsafe += (int64_t)g[(size_t)r * n1 + 5];
    for (int i = 0; i < G; ++i) out->L[i] = fmax(out->L[i], g[(size_t)r * n1 + 6 + i]);
  }
  out->sets.minimizer_var = -INFINITY; out->sets.minimizer_idx = -1;
  if (s2_local) SBO_TRY(sets_pass2(ctx, out->sets.min_ucb0, s2_local));     // reduced with the first gather of the pair stage
  return SBO_OK;
}

extern "C" {

int sbo_comm_unique_id(void* id128) {
  sbo_ctx* ctx = nullptr;
  if (!id128) return sbo_fail(nullptr, SBO_ERR_INVALID, "null id buffer");
  SBO_TRY(nccl_load(nullptr));
  SBO_NCCL(g_nccl.GetUniqueId((ncclUniqueId*)id128));
  return SBO_OK;
}

int sbo_comm_init(sbo_ctx* ctx, int rank, int nranks, const void* id128) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  SBO_REQUIRE(nranks >= 1 && nranks <= 64 && rank >= 0 && rank < nranks && id128, "bad communicator arguments");
  SBO_REQUIRE(ctx->comm == nullptr, "communicator already initialised");
  SBO_TRY(nccl_load(ctx));
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  sbo_comm* cm = new sbo_comm();
  cm->rank = rank; cm->nranks = nranks;
  ncclResult_t r = g_nccl.CommInitRank(&cm->comm, nranks, id, rank);
  if (r != 0) { delete cm; return sbo_fail(ctx, SBO_ERR_CUDA, std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r)); }
  ctx->comm = cm;
  return SBO_OK;
}

int sbo_comm_destroy(sbo_ctx* ctx) {
  if (!ctx || !ctx->comm) return SBO_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  sbo_comm* cm = ctx->comm;
  for (DevBuf* b : {&cm->small, &cm->rows, &cm->vrows, &cm->result, &cm->masks})
    if (b->p) { cudaFree(b->p); b->p = nullptr; b->cap = 0; }
  if (cm->comm) g_nccl.CommDestroy(cm->comm);
  delete cm;
  ctx->comm = nullptr;
  return SBO_OK;
}

int sbo_safeopt_step_sharded(sbo_ctx* ctx, double beta, int mode, int precision, int unsafe_rule, const double* L, sbo_step_result* out) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  SBO_REQUIRE(ctx->comm != nullptr, "sbo_safeopt_step_sharded: call sbo_comm_init first");
  SBO_REQUIRE(out != nullptr, "null result");
  SBO_REQUIRE(mode == SBO_MODE_LIPSCHITZ || mode == SBO_MODE_FANTASY, "bad expander mode");
  memset(out, 0, sizeof(*out));
  const int G = ctx->ms.G;
  const bool fantasy = mode == SBO_MODE_FANTASY;
  const int keep_v = fantasy ? keep_v_of(precision) : 0;
  sbo_sets_result s2;
  SBO_TRY(sharded_sets(ctx, beta, unsafe_rule, (!fantasy && !L) ? 1 : 0, keep_v, &s2, out));
  double Lg[SBO_MAX_G];
  for (int i = 0; i < SBO_MAX_G; ++i) Lg[i] = L ? (i < G ? L[i] : 0.0) : out->L[G - 1];   // SafeOpt.py:110: L of constraint n_fun-1
  SBO_TRY(sharded_pairs(ctx, mode, fantasy ? precision : SBO_PREC_FP64, false, beta, fantasy ? nullptr : Lg, &out->pairs, &s2, &out->sets));
  const double std_min = out->sets.minimizer_idx >= 0 ? sqrt(out->sets.minimizer_var) : 0.0;
  const double std_exp = out->pairs.best_idx >= 0 ? sqrt(out->pairs.best_value) : 0.0;
  out->x_new_idx = std_min > std_exp ? out->sets.minimizer_idx : out->pairs.best_idx;   // test_SafeOpt.py:153-158
  out->explore_idx = -1;
  return SBO_OK;
}

int sbo_goose_step_sharded(sbo_ctx* ctx, double beta, int unsafe_rule, const double* L, sbo_step_result* out) {
  return sbo_goose_step_sharded_ex(ctx, beta, SBO_MODE_LIPSCHITZ, SBO_PREC_FP64, unsafe_rule, L, out);
}

int sbo_goose_step_sharded_ex(sbo_ctx* ctx, double beta, int mode, int precision, int unsafe_rule, const double* L, sbo_step_result* out) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  SBO_REQUIRE(ctx->comm != nullptr, "sbo_goose_step_sharded: call sbo_comm_init first");
  SBO_REQUIRE(out != nullptr, "null result");
  SBO_REQUIRE(mode == SBO_MODE_LIPSCHITZ || mode == SBO_MODE_FANTASY, "bad target mode");
  memset(out, 0, sizeof(*out));
  const int G = ctx->ms.G;
  const bool fantasy = mode == SBO_MODE_FANTASY;
  // fantasy: V rows kept at the GEMM's precision and no gradient, as in sbo_safeopt_step_sharded
  const int keep_v = fantasy ? keep_v_of(precision) : 0;
  SBO_TRY(sharded_sets(ctx, beta, unsafe_rule, (!fantasy && !L) ? 1 : 0, keep_v, nullptr, out));
  double Lg[SBO_MAX_G];
  for (int i = 0; i < SBO_MAX_G; ++i) Lg[i] = L ? (i < G ? L[i] : 0.0) : out->L[G - 1];   // GoOSE.py:100
  SBO_TRY(sharded_pairs(ctx, mode, fantasy ? precision : SBO_PREC_FP64, true, beta, fantasy ? nullptr : Lg, &out->pairs));
  out->explore_idx = -1;
  if (out->sets.min_lcb0 <= out->pairs.best_value || out->pairs.best_idx < 0) {        // test_GoOSE.py:158-162
    out->x_new_idx = out->sets.min_lcb0_idx;
  } else {
    double target[SBO_MAX_D];
    SBO_TRY(sbo_point_coords(ctx, out->pairs.best_idx, target));
    int64_t li; double ld;
    SBO_TRY(argreduce_run(ctx, SBO_ARGMIN_DIST, mask_ptr(ctx, SBO_MASK_SAFE, 0), target, &li, &ld));
    double m[2] = {ld, (double)li};
    std::vector<double> g;
    SBO_TRY(gather_record(ctx, m, 2, g));
    double dv; int64_t di;
    reduce_arg(g, 2, ctx->comm->nranks, 0, false, &dv, &di);
    out->x_new_idx = out->explore_idx = di;
  }
  return SBO_OK;
}

// batch SafeOpt acquisition (batch.cu) on the sharded grid: per pick one all-gather of the ranks' local optima, reduced on the
// raw variances (largest, lowest index on ties) so that every rank commits the same global index
int sbo_safeopt_batch_sharded(sbo_ctx* ctx, int q, sbo_batch_pick* picks, int* n_picked) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  SBO_REQUIRE(ctx->comm != nullptr, "sbo_safeopt_batch_sharded: call sbo_comm_init first");
  SBO_REQUIRE(picks && n_picked, "null result");
  const int R = ctx->comm->nranks;
  SBO_TRY(batch_prepare(ctx, q, nullptr));
  std::vector<double> g;
  int n = 0;
  for (int b = 0; b < q; ++b) {
    BatchRec loc;
    SBO_TRY(batch_local(ctx, &loc));
    double mine[4] = {loc.vmin, (double)loc.imin, loc.vexp, (double)loc.iexp};
    SBO_TRY(gather_record(ctx, mine, 4, g));
    BatchRec r;
    int64_t im, ie;
    reduce_arg(g, 4, R, 0, true, &r.vmin, &im);
    reduce_arg(g, 4, R, 2, true, &r.vexp, &ie);
    r.imin = im; r.iexp = ie;
    const bool hm = r.imin >= 0, he = r.iexp >= 0;
    if (!hm) r.vmin = 0.0;
    if (!he) r.vexp = 0.0;
    const bool take_min = hm && (!he || sqrt(r.vmin) > sqrt(r.vexp));    // test/test_SafeOpt.py:153-158, empty set yields
    r.idx = take_min ? r.imin : r.iexp;
    r.from_exp = (!take_min && he) ? 1 : 0;
    r.pad = 0;
    batch_pick_of(r, &picks[b]);
    if (r.idx < 0) {                                  // M and E are empty on every rank, and stay so
      for (int k = b + 1; k < q; ++k) picks[k] = picks[b];
      break;
    }
    n = b + 1;
    if (b + 1 < q) SBO_TRY(batch_commit(ctx, r.idx));
  }
  stage_changed(ctx, Change::BATCH);
  *n_picked = n;
  return SBO_OK;
}

// batch GoOSE acquisition (batch.cu) on the sharded grid: per pick one all-gather of the ranks' (safe, target) optima, and
// for an explore pick one of their nearest points to the target, both reduced to the smallest value with the lowest global
// index on ties (as sbo_goose_step_sharded_ex), so that every rank commits the same pick
int sbo_goose_batch_sharded(sbo_ctx* ctx, int q, sbo_goose_batch_pick* picks, int* n_picked) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  SBO_REQUIRE(ctx->comm != nullptr, "sbo_goose_batch_sharded: call sbo_comm_init first");
  SBO_REQUIRE(picks && n_picked, "null result");
  const int R = ctx->comm->nranks;
  SBO_TRY(goose_batch_prepare(ctx, q, nullptr));
  std::vector<double> g;
  int n = 0;
  for (int b = 0; b < q; ++b) {
    sbo_goose_batch_pick loc;
    SBO_TRY(goose_batch_local(ctx, &loc));
    double mine[4] = {loc.safe_lcb, (double)loc.safe_idx, loc.target_lcb, (double)loc.target_idx};
    SBO_TRY(gather_record(ctx, mine, 4, g));
    sbo_goose_batch_pick r;
    reduce_arg(g, 4, R, 0, false, &r.safe_lcb, &r.safe_idx);
    reduce_arg(g, 4, R, 2, false, &r.target_lcb, &r.target_idx);
    const bool explore = r.safe_idx >= 0 && r.target_idx >= 0 && !(r.safe_lcb <= r.target_lcb);   // test_GoOSE.py:158-162
    r.explore = explore ? 1 : 0;
    r.pad = 0;
    r.idx = r.safe_idx;
    r.dist = 0.0;
    if (explore) {
      long long li; double ld2;
      SBO_TRY(goose_batch_nearest(ctx, r.target_idx, &li, &ld2));
      double m[2] = {ld2, (double)li};
      SBO_TRY(gather_record(ctx, m, 2, g));
      double d2;
      reduce_arg(g, 2, R, 0, false, &d2, &r.idx);
      r.dist = sqrt(d2);
    }
    picks[b] = r;
    if (r.idx < 0) break;                             // S_b is empty on every rank, and stays so
    n = b + 1;
    if (b + 1 < q) SBO_TRY(goose_batch_commit(ctx, r.idx, explore ? r.target_idx : -1));
  }
  stage_changed(ctx, Change::BATCH);
  *n_picked = n;
  return SBO_OK;
}

}  // extern "C"
