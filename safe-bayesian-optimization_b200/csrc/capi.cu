// capi.cu -- extern "C" entry points of include/sbo_b200.h plus context plumbing.
#include "common.cuh"
#include <math.h>
#include <string.h>

thread_local std::string g_sbo_last_error;

int sbo_fail(sbo_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->err = msg;
  g_sbo_last_error = msg;
  return code;
}

static int ensure(sbo_ctx* ctx, DevBuf& b, size_t bytes, bool headroom) {
  if (bytes == 0) bytes = 16;
  if (b.cap >= bytes) return SBO_OK;
  if (b.p) { cudaStreamSynchronize(ctx->stream); cudaFree(b.p); ctx->mem_now -= (int64_t)b.cap; b.p = nullptr; b.cap = 0; }
  size_t want = headroom ? bytes + bytes / 8 : bytes;
  cudaError_t e = cudaMalloc(&b.p, want);
  if (e != cudaSuccess) { cudaGetLastError(); want = bytes; e = cudaMalloc(&b.p, want); }
  if (e != cudaSuccess) {
    b.p = nullptr; b.cap = 0;
    return sbo_fail(ctx, SBO_ERR_NOMEM, "cudaMalloc of " + std::to_string(bytes) + " bytes failed: " + cudaGetErrorString(e));
  }
  b.cap = want;
  ctx->mem_now += (int64_t)want;
  if (ctx->mem_now > ctx->mem_peak) ctx->mem_peak = ctx->mem_now;
  return SBO_OK;
}
int sbo_ensure(sbo_ctx* ctx, DevBuf& b, size_t bytes) { return ensure(ctx, b, bytes, true); }
int sbo_ensure_exact(sbo_ctx* ctx, DevBuf& b, size_t bytes) { return ensure(ctx, b, bytes, false); }

void sbo_free(sbo_ctx* ctx, DevBuf& b) {
  if (!b.p) return;
  cudaStreamSynchronize(ctx->stream);
  cudaFree(b.p);
  ctx->mem_now -= (int64_t)b.cap;
  b.p = nullptr; b.cap = 0;
}

static void free_buf(DevBuf& b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }

// The one place that decides which stages stay valid.  A change to a stage makes every later stage of the pipeline stale;
// sets pass 2 hangs off pass 1 and makes nothing stale.
void stage_changed(sbo_ctx* ctx, Change c) {
  enum { POST, SETS, PAIRS, BATCH, NONE } stale = NONE;   // the first stage c makes stale; the later ones go with it
  switch (c) {
    case Change::GRID:
      ctx->keep_v = 0;
      [[fallthrough]];
    case Change::MODEL:
      ctx->up.valid = false;
      stale = POST; break;
    case Change::APPEND:             // what sbo_posterior_update is for: ctx->up stays valid
      stale = POST; break;
    case Change::POSTERIOR:
      ctx->keep_v = 0; ctx->up.valid = false;
      stale = POST; break;
    case Change::POSTERIOR_DONE:
      ctx->have_post = true; ctx->have_grad = ctx->up.with_grad;
      ctx->keep_v = ctx->ms.G > 1 ? ctx->up.keep_v : 0;   // V rows exist for the constraints only
      ctx->up.valid = true;
      stale = SETS; break;
    case Change::SETS1:
      ctx->have_sets = true; ctx->have_sets2 = false;
      stale = PAIRS; break;
    case Change::SETS2:
      ctx->have_sets2 = true; break;
    case Change::PAIRS:
      stale = PAIRS; break;
    case Change::PAIRS_PREPARED:
      ctx->ps.prepared = ctx->ps.exportable = true; break;
    case Change::PAIRS_IMPORTED:
      ctx->ps.imported = true; break;
    case Change::EXPANDER:
    case Change::TARGET:             // a batch belongs to the pair stage result it was prepared on
      ctx->have_exp = c == Change::EXPANDER; ctx->have_tgt = c == Change::TARGET;
      stale = BATCH; break;
    case Change::BATCH:
      stale = BATCH; break;
    case Change::BATCH_PREPARED:
      ctx->bt.prepared = true; break;
    case Change::RELEASE_V:          // the update would have to extend rows that are gone, and the export reads them
      if (ctx->keep_v) ctx->up.valid = false;
      ctx->keep_v = 0;
      if (ctx->ps.mode == SBO_MODE_FANTASY) ctx->ps.exportable = false;
      break;
    case Change::RELEASE_PAIRS:      // an unfinished stage loses its operands; the masks of a finished one and a batch stay
      ctx->ps = PairStage{}; break;
  }
  if (stale <= POST) ctx->have_post = ctx->have_grad = false;
  if (stale <= SETS) ctx->have_sets = ctx->have_sets2 = false;
  if (stale <= PAIRS) { ctx->ps = PairStage{}; ctx->have_exp = ctx->have_tgt = false; }
  if (stale <= BATCH) ctx->bt.prepared = false;
}

void ev_begin(sbo_ctx* ctx, int phase) {
  sbo_ctx::EvPair p;
  p.phase = phase;
  for (cudaEvent_t* e : {&p.a, &p.b}) {
    if (!ctx->evpool.empty()) { *e = ctx->evpool.back(); ctx->evpool.pop_back(); }
    else cudaEventCreate(e);
  }
  cudaEventRecord(p.a, ctx->stream);
  ctx->evlog.push_back(p);
}
void ev_end(sbo_ctx* ctx) {
  if (!ctx->evlog.empty()) cudaEventRecord(ctx->evlog.back().b, ctx->stream);
}
void ev_reset(sbo_ctx* ctx, int phase) { ctx->phase_ms[phase] = 0.0; }
void ev_collect(sbo_ctx* ctx) {
  for (auto& p : ctx->evlog) {
    float ms = 0.f;
    if (cudaEventSynchronize(p.b) == cudaSuccess && cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess)
      ctx->phase_ms[p.phase] += ms;
    ctx->evpool.push_back(p.a);
    ctx->evpool.push_back(p.b);
  }
  ctx->evlog.clear();
  cudaGetLastError();
}

extern "C" {

int sbo_version(void) { return 100; }

int sbo_create(int device, sbo_ctx** out) {
  sbo_ctx* ctx = nullptr;
  if (!out) return sbo_fail(nullptr, SBO_ERR_INVALID, "sbo_create: null out pointer");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return sbo_fail(nullptr, SBO_ERR_CUDA, std::string("sbo_create: no CUDA device (") + cudaGetErrorString(e) +
                                               "); this library has no CPU fallback");
  if (device < 0 || device >= ndev) return sbo_fail(nullptr, SBO_ERR_INVALID, "sbo_create: bad device index");
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return sbo_fail(nullptr, SBO_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10)
    return sbo_fail(nullptr, SBO_ERR_CUDA, "sbo_create: device is sm_" + std::to_string(prop.major * 10 + prop.minor) +
                                               ", this library is built for sm_100a (B200) only");
  ctx = new sbo_ctx();
  ctx->device = device;
  e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { delete ctx; return sbo_fail(nullptr, SBO_ERR_CUDA, std::string("cudaStreamCreate: ") + cudaGetErrorString(e)); }
  ctx->own_stream = true;
  *out = ctx;
  return SBO_OK;
}

int sbo_destroy(sbo_ctx* ctx) {
  if (!ctx) return SBO_OK;
  cudaSetDevice(ctx->device);
  sbo_comm_destroy(ctx);
  cudaStreamSynchronize(ctx->stream);
  for (DevBuf* b : {&ctx->Xn, &ctx->Yn, &ctx->alpha, &ctx->W, &ctx->Kmat, &ctx->info, &ctx->pts, &ctx->mean, &ctx->var,
                    &ctx->kx, &ctx->lmax, &ctx->vall, &ctx->tile_bb, &ctx->nll_K, &ctx->nll_in, &ctx->m_safe, &ctx->m_unsafe, &ctx->m_min, &ctx->m_user, &ctx->m_exp,
                    &ctx->m_tgt, &ctx->partials, &ctx->result, &ctx->scan_a, &ctx->scan_b, &ctx->xs_idx, &ctx->zs_idx,
                    &ctx->xs_pay, &ctx->zs_pay, &ctx->hits, &ctx->counts, &ctx->pairctr, &ctx->imp_rows, &ctx->vx, &ctx->vz,
                    &ctx->aux_x, &ctx->aux_z, &ctx->pp_x, &ctx->pp_m, &ctx->pp_v, &ctx->pp_k, &ctx->pp_g, &ctx->tc_row, &ctx->tc_col, &ctx->tc_err, &ctx->exp_rows, &ctx->exp_v, &ctx->key_x, &ctx->key_z, &ctx->perm_x, &ctx->perm_z, &ctx->sort_ws, &ctx->tile_keys, &ctx->item_mask, &ctx->item_list, &ctx->gz_mask, &ctx->gz_idx, &ctx->gz_pay, &ctx->st_score, &ctx->st_mask, &ctx->tabs, &ctx->tc_stats, &ctx->amb_list, &ctx->amb_ctr, &ctx->amb_mask, &ctx->amb_xd, &ctx->amb_zd, &ctx->amb_rx, &ctx->amb_rz, &ctx->amb_pts, &ctx->amb_vx, &ctx->amb_vz, &ctx->amb_rows, &ctx->m_und, &ctx->amb_cell, &ctx->amb_hist, &ctx->amb_tgt,
                    &ctx->bt_mask, &ctx->bt_idx, &ctx->bt_flag, &ctx->bt_v, &ctx->bt_w, &ctx->bt_part, &ctx->bt_pick})
    free_buf(*b);
  ev_collect(ctx);
  for (cudaEvent_t e : ctx->evpool) cudaEventDestroy(e);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return SBO_OK;
}

const char* sbo_last_error(const sbo_ctx* ctx) { return ctx ? ctx->err.c_str() : g_sbo_last_error.c_str(); }

#define ENTER()                                                         \
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context"); \
  cudaSetDevice(ctx->device)

int sbo_set_stream(sbo_ctx* ctx, void* cuda_stream) {
  ENTER();
  cudaStreamSynchronize(ctx->stream);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = (cudaStream_t)cuda_stream;
  ctx->own_stream = false;
  return SBO_OK;
}

int sbo_set_model_ex(sbo_ctx* ctx, int kernel, int n, int d, int G, const double* X_norm, const double* Y_norm,
                     const double* X_mean, const double* X_std, const double* Y_mean, const double* Y_std, const double* hyp) {
  ENTER();
  return model_upload(ctx, kernel, n, d, G, X_norm, Y_norm, X_mean, X_std, Y_mean, Y_std, hyp);
}

int sbo_set_model(sbo_ctx* ctx, int n, int d, int G, const double* X_norm, const double* Y_norm, const double* X_mean,
                  const double* X_std, const double* Y_mean, const double* Y_std, const double* hyp) {
  return sbo_set_model_ex(ctx, SBO_KERNEL_SE, n, d, G, X_norm, Y_norm, X_mean, X_std, Y_mean, Y_std, hyp);
}

int sbo_get_model(sbo_ctx* ctx, double* L, double* W, double* alpha) {
  ENTER();
  SBO_REQUIRE(ctx->have_model, "no model");
  const int n = ctx->ms.n, np = ctx->ms.npad, G = ctx->ms.G;
  std::vector<double> tmp((size_t)np * np);
  for (int g = 0; g < G; ++g) {
    for (int which = 0; which < 2; ++which) {
      double* dst = which == 0 ? L : W;
      if (!dst) continue;
      const double* src = (const double*)(which == 0 ? ctx->Kmat.p : ctx->W.p) + (size_t)g * np * np;
      SBO_CUDA(cudaMemcpyAsync(tmp.data(), src, sizeof(double) * tmp.size(), cudaMemcpyDeviceToHost, ctx->stream));
      SBO_CUDA(cudaStreamSynchronize(ctx->stream));
      for (int r = 0; r < n; ++r)
        for (int c = 0; c < n; ++c) dst[((size_t)g * n + r) * n + c] = (c <= r) ? tmp[(size_t)r * np + c] : 0.0;
    }
    if (alpha) {
      SBO_CUDA(cudaMemcpyAsync(alpha + (size_t)g * n, (const double*)ctx->alpha.p + (size_t)g * np, sizeof(double) * n,
                               cudaMemcpyDeviceToHost, ctx->stream));
      SBO_CUDA(cudaStreamSynchronize(ctx->stream));
    }
  }
  return SBO_OK;
}

int sbo_set_grid(sbo_ctx* ctx, int d, const int64_t* pts_per_dim, const double* lo, const double* hi) {
  ENTER();
  SBO_REQUIRE(d >= 1 && d <= SBO_MAX_D, "d out of range (1..8)");
  SBO_REQUIRE(pts_per_dim && lo && hi, "null grid pointer");
  GridSpec g{};
  g.kind = 1; g.d = d;
  long long N = 1;
  for (int k = 0; k < d; ++k) {
    SBO_REQUIRE(pts_per_dim[k] >= 1, "pts_per_dim must be >= 1");
    g.pts[k] = pts_per_dim[k];
    g.stride[k] = N;
    g.lo[k] = lo[k]; g.hi[k] = hi[k];
    g.step[k] = pts_per_dim[k] > 1 ? (hi[k] - lo[k]) / (double)(pts_per_dim[k] - 1) : 0.0;   // numpy.linspace step
    SBO_REQUIRE(N <= (1LL << 40) / pts_per_dim[k], "grid too large");
    N *= pts_per_dim[k];
  }
  for (int k = d; k < SBO_MAX_D; ++k) { g.pts[k] = 1; g.stride[k] = N; }
  g.N = N; g.first = 0; g.count = N;
  ctx->gs = g;
  ctx->have_grid = true;
  stage_changed(ctx, Change::GRID);
  return SBO_OK;
}

int sbo_set_points(sbo_ctx* ctx, int64_t N, int d, const double* pts) {
  ENTER();
  SBO_REQUIRE(d >= 1 && d <= SBO_MAX_D, "d out of range (1..8)");
  SBO_REQUIRE(N >= 1 && pts, "bad points");
  SBO_TRY(sbo_ensure(ctx, ctx->pts, sizeof(double) * (size_t)N * d));
  SBO_CUDA(cudaMemcpyAsync(ctx->pts.p, pts, sizeof(double) * (size_t)N * d, cudaMemcpyHostToDevice, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  GridSpec g{};
  g.kind = 2; g.d = d; g.N = N; g.first = 0; g.count = N;
  g.explicit_pts = (const double*)ctx->pts.p;
  ctx->gs = g;
  ctx->have_grid = true;
  stage_changed(ctx, Change::GRID);
  return SBO_OK;
}

int sbo_set_shard(sbo_ctx* ctx, int64_t first, int64_t count) {
  ENTER();
  SBO_REQUIRE(ctx->have_grid, "sbo_set_shard: no grid");
  SBO_REQUIRE(first >= 0 && count >= 1 && first + count <= ctx->gs.N, "shard out of range");
  ctx->gs.first = first; ctx->gs.count = count;
  ctx->gs.cyc_n = 0; ctx->gs.cyc_rank = 0; ctx->gs.cyc_blk = 0;
  stage_changed(ctx, Change::GRID);
  return SBO_OK;
}

int sbo_set_shard_cyclic(sbo_ctx* ctx, int rank, int nranks, int64_t block, int64_t* count_out) {
  ENTER();
  SBO_REQUIRE(ctx->have_grid, "sbo_set_shard_cyclic: no grid");
  SBO_REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks && block >= 32 && block % 32 == 0, "bad cyclic shard");
  GridSpec& g = ctx->gs;
  const long long nblk = cdiv(g.N, block);
  long long count = 0;
  for (long long sb = 0; sb * nranks < nblk; ++sb) {      // same slot rule as shard_global()
    const long long b = sb * nranks + (rank + sb + sb / nranks + sb / ((long long)nranks * nranks)) % nranks;
    if (b < nblk) count += (b == nblk - 1) ? (g.N - b * block) : block;
  }
  SBO_REQUIRE(count >= 1, "this rank owns no grid points");
  g.first = 0; g.count = count;
  g.cyc_n = nranks; g.cyc_rank = rank; g.cyc_blk = block;
  if (nranks == 1) { g.cyc_n = 0; }
  if (count_out) *count_out = count;
  stage_changed(ctx, Change::GRID);
  return SBO_OK;
}

int sbo_point_coords(sbo_ctx* ctx, int64_t p, double* x) {
  ENTER();
  SBO_REQUIRE(ctx->have_grid && x, "no grid");
  const GridSpec& g = ctx->gs;
  SBO_REQUIRE(p >= 0 && p < g.N, "point index out of range");
  if (g.kind == 1) {
    for (int k = 0; k < g.d; ++k) {
      const long long i = (p / g.stride[k]) % g.pts[k];
      x[k] = (g.pts[k] > 1 && i == g.pts[k] - 1) ? g.hi[k] : ((double)i * g.step[k] + g.lo[k]);
    }
  } else {
    SBO_CUDA(cudaMemcpyAsync(x, g.explicit_pts + (size_t)p * g.d, sizeof(double) * g.d, cudaMemcpyDeviceToHost, ctx->stream));
    SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return SBO_OK;
}

int sbo_posterior(sbo_ctx* ctx, int with_grad, int keep_v, double* mean, double* var) {
  ENTER();
  SBO_TRY(posterior_run(ctx, with_grad, keep_v));
  const size_t bytes = sizeof(double) * (size_t)ctx->ms.G * ctx->gs.count;
  if (mean) SBO_CUDA(cudaMemcpyAsync(mean, ctx->mean.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (var) SBO_CUDA(cudaMemcpyAsync(var, ctx->var.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  ev_collect(ctx);
  return SBO_OK;
}

int sbo_posterior_update(sbo_ctx* ctx, double* mean, double* var, sbo_update_info* info) {
  ENTER();
  sbo_update_info tmp;
  SBO_TRY(posterior_update(ctx, info ? info : &tmp));
  const size_t bytes = sizeof(double) * (size_t)ctx->ms.G * ctx->gs.count;
  if (mean) SBO_CUDA(cudaMemcpyAsync(mean, ctx->mean.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (var) SBO_CUDA(cudaMemcpyAsync(var, ctx->var.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  ev_collect(ctx);
  return SBO_OK;
}

int sbo_point_posterior(sbo_ctx* ctx, int64_t m, const double* x, double* mean, double* var) {
  ENTER();
  return posterior_points(ctx, m, x, mean, var);
}

int sbo_point_mean_grad(sbo_ctx* ctx, int gp, int64_t m, const double* x, double* grad) {
  ENTER();
  SBO_REQUIRE(grad != nullptr, "null grad");
  return posterior_point_grad(ctx, gp, m, x, grad);
}

int sbo_lipschitz(sbo_ctx* ctx, double* L) {
  ENTER();
  SBO_REQUIRE(ctx->have_post && ctx->have_grad && L, "sbo_lipschitz: call sbo_posterior(with_grad=1) first");
  SBO_CUDA(cudaMemcpyAsync(L, ctx->lmax.p, sizeof(double) * ctx->ms.G, cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}

int sbo_sets_pass1(sbo_ctx* ctx, double beta, int unsafe_rule, int strict, sbo_sets_result* out) {
  ENTER();
  return sets_pass1(ctx, beta, unsafe_rule, strict, out);
}
int sbo_sets_pass2(sbo_ctx* ctx, double min_ucb0, sbo_sets_result* out) {
  ENTER();
  return sets_pass2(ctx, min_ucb0, out);
}
int sbo_sets(sbo_ctx* ctx, double beta, int unsafe_rule, int strict, sbo_sets_result* out) {
  ENTER();
  sbo_sets_result r1, r2;
  SBO_TRY(sets_pass1(ctx, beta, unsafe_rule, strict, &r1));
  SBO_TRY(sets_pass2(ctx, r1.min_ucb0, &r2));
  if (out) *out = r2;
  return SBO_OK;
}

int sbo_get_mask(sbo_ctx* ctx, int mask_kind, int which, uint32_t* words) {
  ENTER();
  SBO_REQUIRE(ctx->have_sets && words, "sbo_get_mask: no sets");
  SBO_REQUIRE(mask_kind != SBO_MASK_MIN || ctx->have_sets2, "minimiser mask needs sbo_sets_pass2");
  SBO_REQUIRE(which >= 0 && which < SBO_MAX_G, "bad mask index");
  const uint32_t* p = mask_ptr(ctx, mask_kind, which);
  SBO_REQUIRE(p != nullptr, "mask not available");
  SBO_CUDA(cudaMemcpyAsync(words, p, sizeof(uint32_t) * mask_words(ctx), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}

int sbo_set_user_mask(sbo_ctx* ctx, const uint32_t* words) {
  ENTER();
  SBO_REQUIRE(ctx->have_grid && words, "sbo_set_user_mask: no grid");
  SBO_TRY(sbo_ensure(ctx, ctx->m_user, sizeof(uint32_t) * mask_words(ctx)));
  SBO_CUDA(cudaMemcpyAsync(ctx->m_user.p, words, sizeof(uint32_t) * mask_words(ctx), cudaMemcpyHostToDevice, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}

int sbo_user_mask_ball(sbo_ctx* ctx, int mask_kind, const double* x0, double r) {
  ENTER();
  return ball_mask(ctx, mask_kind, x0, r);
}

int sbo_mask_dev(sbo_ctx* ctx, int mask_kind, int which, void** dev_ptr, int64_t* n_words) {
  ENTER();
  SBO_REQUIRE(dev_ptr && n_words, "null out pointer");
  uint32_t* p = mask_ptr(ctx, mask_kind, which);
  SBO_REQUIRE(p != nullptr, "mask not available");
  *dev_ptr = p; *n_words = mask_words(ctx);
  return SBO_OK;
}

int sbo_posterior_dev(sbo_ctx* ctx, void** mean_dev, void** var_dev) {
  ENTER();
  SBO_REQUIRE(ctx->have_post, "no posterior");
  if (mean_dev) *mean_dev = ctx->mean.p;
  if (var_dev) *var_dev = ctx->var.p;
  return SBO_OK;
}

int sbo_argreduce(sbo_ctx* ctx, int reduce_kind, int mask_kind, int which, const double* target, int64_t* idx, double* value) {
  ENTER();
  SBO_REQUIRE(ctx->have_sets || mask_kind == SBO_MASK_USER, "sbo_argreduce: no sets");
  return argreduce_run(ctx, reduce_kind, mask_ptr(ctx, mask_kind, which), target, idx, value);
}

int sbo_expander(sbo_ctx* ctx, int mode, int precision, double beta, const double* L, sbo_pair_result* out, int32_t* counts) {
  ENTER();
  if (mode == SBO_MODE_LIPSCHITZ) return pairs_lipschitz(ctx, false, beta, L, out);
  if (mode == SBO_MODE_FANTASY) return pairs_fantasy(ctx, precision, beta, out, counts);
  return sbo_fail(ctx, SBO_ERR_INVALID, "bad expander mode");
}

int sbo_goose_target(sbo_ctx* ctx, double beta, const double* L, sbo_pair_result* out) {
  return sbo_goose_target_ex(ctx, SBO_MODE_LIPSCHITZ, SBO_PREC_FP64, beta, L, out);
}

int sbo_goose_target_ex(sbo_ctx* ctx, int mode, int precision, double beta, const double* L, sbo_pair_result* out) {
  ENTER();
  if (mode == SBO_MODE_LIPSCHITZ) return pairs_lipschitz(ctx, true, beta, L, out);
  if (mode == SBO_MODE_FANTASY) return pairs_goose_fantasy(ctx, precision, beta, out);
  return sbo_fail(ctx, SBO_ERR_INVALID, "bad target mode");
}

int sbo_pairs_prepare(sbo_ctx* ctx, int mode, int precision, double beta, const double* L, sbo_pairs_info* info) {
  ENTER();
  return pairs_prepare(ctx, mode, precision, beta, L, info);
}
int sbo_pairs_export_dev(sbo_ctx* ctx, void* rows_dev, void* vrows_dev) {
  ENTER();
  SBO_TRY(pairs_export(ctx, rows_dev, vrows_dev));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}
int sbo_pairs_import_dev(sbo_ctx* ctx, int64_t n_total, const void* rows_dev, const void* vrows_dev) {
  ENTER();
  return pairs_import(ctx, n_total, rows_dev, vrows_dev);
}
int sbo_pairs_set_segments(sbo_ctx* ctx, int nranks, int rank, const int64_t* n_per_rank) {
  ENTER();
  return pairs_set_segments(ctx, nranks, rank, n_per_rank);
}
int sbo_pairs_set_global_unsafe_dev(sbo_ctx* ctx, const void* gathered_words_dev, int64_t words_per_rank, int nranks) {
  ENTER();
  return pairs_set_global_unsafe(ctx, gathered_words_dev, words_per_rank, nranks);
}
int sbo_mask_export_dev(sbo_ctx* ctx, int mask_kind, int which, void* dst_dev, int64_t dst_words) {
  ENTER();
  SBO_REQUIRE(ctx->have_sets && dst_dev, "sbo_mask_export_dev: no sets");
  const uint32_t* p = mask_ptr(ctx, mask_kind, which);
  SBO_REQUIRE(p != nullptr, "mask not available");
  const long long nw = mask_words(ctx);
  SBO_REQUIRE(dst_words >= nw, "destination too small");
  SBO_CUDA(cudaMemcpyAsync(dst_dev, p, sizeof(uint32_t) * (size_t)nw, cudaMemcpyDeviceToDevice, ctx->stream));
  if (dst_words > nw) SBO_CUDA(cudaMemsetAsync((uint32_t*)dst_dev + nw, 0, sizeof(uint32_t) * (size_t)(dst_words - nw), ctx->stream));
  return SBO_OK;
}
int sbo_pairs_run_dev(sbo_ctx* ctx, int goose, void* result_dev) {
  ENTER();
  SBO_TRY(pairs_run(ctx, goose, result_dev));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}
int sbo_pairs_finish_dev(sbo_ctx* ctx, int goose, int64_t offset, const void* result_dev, sbo_pair_result* out, int32_t* counts) {
  ENTER();
  return pairs_finish(ctx, goose, offset, result_dev, out, counts);
}

int64_t sbo_kernel_launches(sbo_ctx* ctx, int reset) {
  if (!ctx) return 0;
  const int64_t v = ctx->launches;
  if (reset) ctx->launches = 0;
  return v;
}

int64_t sbo_mem_peak(sbo_ctx* ctx, int reset) {
  if (!ctx) return 0;
  const int64_t v = ctx->mem_peak;
  if (reset) ctx->mem_peak = ctx->mem_now;
  return v;
}

int sbo_refine_stats(sbo_ctx* ctx, int64_t* cells, int64_t* fp64_rows) {
  ENTER();
  SBO_REQUIRE(cells && fp64_rows, "null out pointer");
  *cells = ctx->refine_cells; *fp64_rows = ctx->refine_rows;
  return SBO_OK;
}

int sbo_phase_ms(sbo_ctx* ctx, int phase, double* ms) {
  ENTER();
  SBO_REQUIRE(phase >= 0 && phase < 9 && ms, "bad phase");
  *ms = ctx->phase_ms[phase];
  return SBO_OK;
}

int sbo_nll_batch_ex(sbo_ctx* ctx, int kernel, int n, int d, const double* X_norm, const double* y, int P, const double* hyp,
                     double* nll) {
  ENTER();
  return nll_batch(ctx, kernel, n, d, X_norm, y, P, hyp, nll);
}

int sbo_nll_batch(sbo_ctx* ctx, int n, int d, const double* X_norm, const double* y, int P, const double* hyp, double* nll) {
  return sbo_nll_batch_ex(ctx, SBO_KERNEL_SE, n, d, X_norm, y, P, hyp, nll);
}

int sbo_append_sample(sbo_ctx* ctx, const double* x_norm_new, const double* y_norm_new) {
  ENTER();
  return model_append(ctx, x_norm_new, y_norm_new);
}

int sbo_stable_minmax(sbo_ctx* ctx, int n_controlled, int fun_kind, double beta, int64_t* xc_idx, double* value,
                      int64_t* n_robust_safe, double* score) {
  ENTER();
  return stable_minmax(ctx, n_controlled, fun_kind, beta, xc_idx, value, n_robust_safe, score);
}

int sbo_release(sbo_ctx* ctx, int what) {
  ENTER();
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  if (what & 1) {
    stage_changed(ctx, Change::RELEASE_V);
    ctx->mem_now -= (int64_t)ctx->vall.cap; free_buf(ctx->vall);
  }
  if (what & 2) {
    for (DevBuf* b : {&ctx->vx, &ctx->vz, &ctx->exp_v, &ctx->tc_row, &ctx->tc_col, &ctx->imp_rows}) { ctx->mem_now -= (int64_t)b->cap; free_buf(*b); }
    // workspaces of the FP64 refinement: the ambiguous-pair list, its points, rank maps, buckets and FP64 rows
    for (DevBuf* b : {&ctx->amb_list, &ctx->amb_mask, &ctx->amb_xd, &ctx->amb_zd, &ctx->amb_rx, &ctx->amb_rz, &ctx->amb_pts,
                      &ctx->amb_vx, &ctx->amb_vz, &ctx->amb_cell, &ctx->amb_hist, &ctx->amb_tgt})
      sbo_free(ctx, *b);
    stage_changed(ctx, Change::RELEASE_PAIRS);
  }
  return SBO_OK;
}

int sbo_set_option(sbo_ctx* ctx, const char* name, int64_t value) {
  ENTER();
  SBO_REQUIRE(name != nullptr, "null option name");
  if (!strcmp(name, "posterior_variant")) { ctx->opt_posterior_variant = value; return SBO_OK; }
  if (!strcmp(name, "posterior_tables")) { ctx->opt_posterior_tables = value; return SBO_OK; }
  if (!strcmp(name, "posterior_fused")) { ctx->opt_posterior_fused = value; return SBO_OK; }
  if (!strcmp(name, "posterior_chunk_mb")) { ctx->opt_posterior_chunk_mb = value; return SBO_OK; }
  if (!strcmp(name, "fantasy_variant")) { ctx->opt_fantasy_variant = value; return SBO_OK; }
  if (!strcmp(name, "prior_mean_zero")) { ctx->opt_prior_mean_zero = value; return SBO_OK; }
  if (!strcmp(name, "fantasy_refine_cap")) { ctx->opt_fantasy_refine_cap = value; return SBO_OK; }
  if (!strcmp(name, "fantasy_refine")) { ctx->opt_fantasy_refine = value; return SBO_OK; }
  if (!strcmp(name, "fantasy_refine_mb")) {
    SBO_REQUIRE(value >= 0, "fantasy_refine_mb must be >= 0 (0 = the free device memory)");
    ctx->opt_fantasy_refine_mb = value; return SBO_OK;
  }
  if (!strcmp(name, "fantasy_f64_variant")) { ctx->opt_fantasy_f64_variant = value; return SBO_OK; }
  if (!strcmp(name, "pair_cull")) { ctx->opt_pair_cull = value; return SBO_OK; }
  if (!strcmp(name, "fantasy_gx")) { ctx->opt_fantasy_gx = value; return SBO_OK; }
  if (!strcmp(name, "fantasy_prune")) { ctx->opt_fantasy_prune = value; return SBO_OK; }
  return sbo_fail(ctx, SBO_ERR_INVALID, std::string("unknown option ") + name);
}

}  // extern "C"
