// model.cu -- model upload: K_i = k_i(X, X) + (sn2+eps_f32) I (SE or Matern, common.cuh), blocked Cholesky K = L L^T,
// W = L^-1 (lower-triangular inverse) and alpha = K^-1 (Y_i - m0_i), all FP64 on the device.
// Replaces the host-side jnp.linalg.inv(Kopt) of models/GP_Safe.py:226-232 for the grid path.
#include "common.cuh"
#include <math.h>
#include <string.h>

#define NB 32   // factorisation block size

// K[g][r][c], padded to npad: identity on the padded diagonal so the padded matrix stays SPD.
template <class KC>
__global__ void k_build_K(ModelSpec ms, double* __restrict__ K) {
  const KC kc(ms.kernel);
  const int g = blockIdx.z;
  const int r = blockIdx.y * blockDim.y + threadIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= ms.npad || c >= ms.npad) return;
  double v;
  if (r < ms.n && c < ms.n) {
    double s = 0.0;
    for (int k = 0; k < ms.d; ++k) {
      const double df = ms.Xn[r * ms.d + k] - ms.Xn[c * ms.d + k];
      s += df * df * ms.inv_ell[g][k];
    }
    v = kc.value(s, ms.sf2[g]);
    if (r == c) v += ms.sn2[g];
  } else {
    v = (r == c) ? 1.0 : 0.0;
  }
  K[((size_t)g * ms.npad + r) * ms.npad + c] = v;
}

// factor the NBxNB diagonal block kb in shared memory (right-looking, unblocked)
__global__ void __launch_bounds__(NB * NB) k_chol_diag(double* __restrict__ A, int npad, int kb, int* __restrict__ info) {
  __shared__ double a[NB][NB + 1];
  const int g = blockIdx.x;
  double* Ag = A + (size_t)g * npad * npad;
  const int tx = threadIdx.x, ty = threadIdx.y;   // ty = row, tx = col
  const int o = kb * NB;
  a[ty][tx] = Ag[(size_t)(o + ty) * npad + o + tx];
  __syncthreads();
  for (int j = 0; j < NB; ++j) {
    if (tx == j && ty == j) {
      const double p = a[j][j];
      if (!(p > 0.0)) { atomicExch(info + g, o + j + 1); a[j][j] = 1.0; }
      else a[j][j] = sqrt(p);
    }
    __syncthreads();
    if (tx == j && ty > j) a[ty][j] /= a[j][j];
    __syncthreads();
    if (tx > j && ty >= tx) a[ty][tx] -= a[ty][j] * a[tx][j];
    __syncthreads();
  }
  Ag[(size_t)(o + ty) * npad + o + tx] = (tx <= ty) ? a[ty][tx] : 0.0;
}

// panel below the diagonal block:  X * Lkk^T = A_panel   (one thread per row)
__global__ void __launch_bounds__(128) k_chol_panel(double* __restrict__ A, int npad, int kb) {
  __shared__ double l[NB][NB + 1];
  const int g = blockIdx.y;
  double* Ag = A + (size_t)g * npad * npad;
  const int o = kb * NB;
  for (int e = threadIdx.x; e < NB * NB; e += blockDim.x) l[e / NB][e % NB] = Ag[(size_t)(o + e / NB) * npad + o + e % NB];
  __syncthreads();
  const int row = o + NB + blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= npad) return;
  double x[NB];
#pragma unroll
  for (int j = 0; j < NB; ++j) x[j] = Ag[(size_t)row * npad + o + j];
#pragma unroll
  for (int j = 0; j < NB; ++j) {
    double s = x[j];
#pragma unroll
    for (int t = 0; t < j; ++t) s -= x[t] * l[j][t];
    x[j] = s / l[j][j];
  }
#pragma unroll
  for (int j = 0; j < NB; ++j) Ag[(size_t)row * npad + o + j] = x[j];
}

// trailing update  A[bi][bj] -= P_bi * P_bj^T  for lower tiles bi >= bj (NBxNB tiles)
__global__ void __launch_bounds__(NB * NB) k_chol_update(double* __restrict__ A, int npad, int kb) {
  const int bj = blockIdx.x, bi = blockIdx.y;
  if (bj > bi) return;
  __shared__ double pi[NB][NB + 1], pj[NB][NB + 1];
  const int g = blockIdx.z;
  double* Ag = A + (size_t)g * npad * npad;
  const int o = kb * NB;
  const int r0 = o + NB + bi * NB, c0 = o + NB + bj * NB;
  const int tx = threadIdx.x, ty = threadIdx.y;
  pi[ty][tx] = Ag[(size_t)(r0 + ty) * npad + o + tx];
  pj[ty][tx] = Ag[(size_t)(c0 + ty) * npad + o + tx];
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int t = 0; t < NB; ++t) s += pi[ty][t] * pj[tx][t];
  Ag[(size_t)(r0 + ty) * npad + c0 + tx] -= s;
}

// inverse of each NBxNB lower-triangular diagonal block of L -> diagonal blocks of W
__global__ void __launch_bounds__(NB) k_tri_diag_inv(const double* __restrict__ A, double* __restrict__ W, int npad) {
  __shared__ double l[NB][NB + 1];
  const int kb = blockIdx.x, g = blockIdx.y;
  const double* Ag = A + (size_t)g * npad * npad;
  double* Wg = W + (size_t)g * npad * npad;
  const int o = kb * NB;
  for (int e = threadIdx.x; e < NB * NB; e += NB) l[e / NB][e % NB] = Ag[(size_t)(o + e / NB) * npad + o + e % NB];
  __syncthreads();
  const int c = threadIdx.x;   // column of the inverse: solve L x = e_c
  double x[NB];
#pragma unroll
  for (int r = 0; r < NB; ++r) {
    double s = (r == c) ? 1.0 : 0.0;
#pragma unroll
    for (int t = 0; t < r; ++t) s -= l[r][t] * x[t];
    x[r] = (r < c) ? 0.0 : s / l[r][r];
  }
#pragma unroll
  for (int r = 0; r < NB; ++r) Wg[(size_t)(o + r) * npad + o + c] = x[r];
}

// column block k of W = L^-1 by block forward substitution (one CTA per column block):
//   W_ik = -W_ii * sum_{j=k}^{i-1} L_ij W_jk ,  i = k+1 .. nblk-1
__global__ void __launch_bounds__(NB * NB) k_tri_inv_cols(const double* __restrict__ A, double* __restrict__ W, int npad) {
  __shared__ double sa[NB][NB + 1], sb[NB][NB + 1];
  const int k = blockIdx.x, g = blockIdx.y;
  const int nblk = npad / NB;
  const double* Ag = A + (size_t)g * npad * npad;
  double* Wg = W + (size_t)g * npad * npad;
  const int tx = threadIdx.x, ty = threadIdx.y;
  for (int i = k + 1; i < nblk; ++i) {
    double t = 0.0;
    for (int j = k; j < i; ++j) {
      sa[ty][tx] = Ag[(size_t)(i * NB + ty) * npad + j * NB + tx];   // L_ij
      sb[ty][tx] = Wg[(size_t)(j * NB + ty) * npad + k * NB + tx];   // W_jk (written by this CTA earlier)
      __syncthreads();
#pragma unroll
      for (int q = 0; q < NB; ++q) t += sa[ty][q] * sb[q][tx];
      __syncthreads();
    }
    sa[ty][tx] = Wg[(size_t)(i * NB + ty) * npad + i * NB + tx];     // W_ii
    sb[ty][tx] = t;
    __syncthreads();
    double r = 0.0;
#pragma unroll
    for (int q = 0; q < NB; ++q) r += sa[ty][q] * sb[q][tx];
    Wg[(size_t)(i * NB + ty) * npad + k * NB + tx] = -r;
    __syncthreads();   // make W_ik visible to the whole CTA before the next block row reads it
  }
}

// alpha = W^T (W (y - m0))
__global__ void __launch_bounds__(256) k_alpha(ModelSpec ms, const double* __restrict__ Yn, double* __restrict__ tmp,
                                               double* __restrict__ alpha) {
  const int g = blockIdx.x;
  const int np = ms.npad;
  const double* Wg = ms.W + (size_t)g * np * np;
  double* t = tmp + (size_t)g * np;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  for (int r = warp; r < np; r += nwarp) {   // one warp per row: coalesced reads of W[r][0..r]
    double s = 0.0;
    for (int c = lane; c <= r && c < ms.n; c += 32) s += Wg[(size_t)r * np + c] * (Yn[(size_t)c * ms.G + g] - ms.m0[g]);
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
    if (lane == 0) t[r] = (r < ms.n) ? s : 0.0;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < np; c += blockDim.x) {
    double s = 0.0;
    for (int r = c; r < ms.n; ++r) s += Wg[(size_t)r * np + c] * t[r];
    alpha[(size_t)g * np + c] = (c < ms.n) ? s : 0.0;
  }
}

int model_upload(sbo_ctx* ctx, int kernel, int n, int d, int G, const double* X_norm, const double* Y_norm,
                 const double* X_mean, const double* X_std, const double* Y_mean, const double* Y_std,
                 const double* hyp) {
  SBO_REQUIRE(n >= 1 && n <= 16384, "n out of range");
  SBO_REQUIRE(d >= 1 && d <= SBO_MAX_D, "d out of range (1..8)");
  SBO_REQUIRE(G >= 1 && G <= SBO_MAX_G, "G out of range (1..8)");
  SBO_REQUIRE(X_norm && Y_norm && X_mean && X_std && Y_mean && Y_std && hyp, "null model pointer");
  SBO_REQUIRE(kernel_valid(kernel), "unknown kernel (SBO_KERNEL_SE, SBO_KERNEL_MATERN32 or SBO_KERNEL_MATERN52)");
  // a refused argument leaves the installed model and every stage built on it untouched; from here on the old model is
  // overwritten, so it and everything after it is invalid until this upload succeeds
  ctx->have_model = false;
  stage_changed(ctx, Change::MODEL);
  ev_reset(ctx, 0);
  ev_begin(ctx, 0);
  ModelSpec& ms = ctx->ms;
  memset(&ms, 0, sizeof(ms));
  ms.n = n; ms.d = d; ms.G = G; ms.kernel = kernel;
  ms.npad = (int)(cdiv(n, 128) * 128);   // multiple of the 128-row blocks of the DMMA solve kernel
  const int np = ms.npad;
  for (int k = 0; k < d; ++k) { ms.Xmean[k] = X_mean[k]; ms.Xstd[k] = X_std[k]; }
  for (int g = 0; g < G; ++g) {
    ms.Ymean[g] = Y_mean[g]; ms.Ystd[g] = Y_std[g];
    // GP_Safe.py:331-332; option prior_mean_zero: the zero prior of GP_Robust.py:322-323 (StableOpt's model)
    ms.m0[g] = (g == 0 || ctx->opt_prior_mean_zero) ? 0.0 : (-2.0 * Y_mean[g]) / Y_std[g];
    for (int k = 0; k < d; ++k) ms.inv_ell[g][k] = 1.0 / exp(2.0 * hyp[(size_t)k * G + g]);   // :338
    ms.sf2[g] = exp(2.0 * hyp[(size_t)d * G + g]);
    ms.sn2[g] = exp(2.0 * hyp[(size_t)(d + 1) * G + g]) + SBO_EPS_F32;         // :229
  }
  SBO_TRY(sbo_ensure(ctx, ctx->Xn, sizeof(double) * np * d));
  SBO_TRY(sbo_ensure(ctx, ctx->Yn, sizeof(double) * (size_t)n * G));
  SBO_TRY(sbo_ensure(ctx, ctx->alpha, sizeof(double) * (size_t)G * np * 2));
  SBO_TRY(sbo_ensure(ctx, ctx->W, sizeof(double) * (size_t)G * np * np));
  SBO_TRY(sbo_ensure(ctx, ctx->Kmat, sizeof(double) * (size_t)G * np * np));
  SBO_TRY(sbo_ensure(ctx, ctx->info, sizeof(int) * SBO_MAX_G));
  SBO_CUDA(cudaMemsetAsync(ctx->Xn.p, 0, sizeof(double) * np * d, ctx->stream));
  SBO_CUDA(cudaMemcpyAsync(ctx->Xn.p, X_norm, sizeof(double) * (size_t)n * d, cudaMemcpyHostToDevice, ctx->stream));
  SBO_CUDA(cudaMemcpyAsync(ctx->Yn.p, Y_norm, sizeof(double) * (size_t)n * G, cudaMemcpyHostToDevice, ctx->stream));
  SBO_CUDA(cudaMemsetAsync(ctx->W.p, 0, sizeof(double) * (size_t)G * np * np, ctx->stream));
  SBO_CUDA(cudaMemsetAsync(ctx->info.p, 0, sizeof(int) * SBO_MAX_G, ctx->stream));
  ms.Xn = (const double*)ctx->Xn.p;
  ms.alpha = (const double*)ctx->alpha.p;
  ms.W = (const double*)ctx->W.p;
  double* K = (double*)ctx->Kmat.p;
  double* W = (double*)ctx->W.p;

  {
    dim3 b(16, 16), g((unsigned)cdiv(np, 16), (unsigned)cdiv(np, 16), (unsigned)G);
    with_kernel(kernel, [&](auto kc) { k_build_K<decltype(kc)><<<g, b, 0, ctx->stream>>>(ms, K); });
    SBO_LAUNCH_CHECK();
  }
  const int nblk = np / NB;
  for (int kb = 0; kb < nblk; ++kb) {
    k_chol_diag<<<G, dim3(NB, NB), 0, ctx->stream>>>(K, np, kb, (int*)ctx->info.p);
    SBO_LAUNCH_CHECK();
    const int below = np - (kb + 1) * NB;
    if (below > 0) {
      k_chol_panel<<<dim3((unsigned)cdiv(below, 128), (unsigned)G), 128, 0, ctx->stream>>>(K, np, kb);
      SBO_LAUNCH_CHECK();
      const int nb = below / NB;
      k_chol_update<<<dim3(nb, nb, G), dim3(NB, NB), 0, ctx->stream>>>(K, np, kb);
      SBO_LAUNCH_CHECK();
    }
  }
  k_tri_diag_inv<<<dim3(nblk, G), NB, 0, ctx->stream>>>(K, W, np);
  SBO_LAUNCH_CHECK();
  k_tri_inv_cols<<<dim3(nblk, G), dim3(NB, NB), 0, ctx->stream>>>(K, W, np);
  SBO_LAUNCH_CHECK();
  k_alpha<<<G, 256, 0, ctx->stream>>>(ms, (const double*)ctx->Yn.p, (double*)ctx->alpha.p + (size_t)G * np,
                                       (double*)ctx->alpha.p);
  SBO_LAUNCH_CHECK();
  int info[SBO_MAX_G];
  SBO_CUDA(cudaMemcpyAsync(info, ctx->info.p, sizeof(int) * SBO_MAX_G, cudaMemcpyDeviceToHost, ctx->stream));
  ev_end(ctx);
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  ev_collect(ctx);
  for (int g = 0; g < G; ++g)
    if (info[g] != 0)
      return sbo_fail(ctx, SBO_ERR_NUMERIC, "K of GP " + std::to_string(g) + " is not positive definite at pivot " +
                                                std::to_string(info[g] - 1));
  ctx->have_model = true;
  return SBO_OK;
}


// =============================================================================================
// Rank-1 append (SURVEY.md section 8f row 1): one new observation at FIXED hyper-parameters and FIXED normalisation.
// The reference's add_sample (GP_Safe.py:283-304) re-fits and re-normalises, i.e. rebuilds K and inv(K) from scratch
// (O(n^3)); at fixed hyper-parameters the factor only gains one row:
//   l = L^-1 k_new = W k_new ,  l_nn = sqrt(k(x,x) + sn2 - |l|^2) ,  L' = [[L, 0], [l^T, l_nn]] ,
//   W' = L'^-1 = [[W, 0], [-(l^T W)/l_nn, 1/l_nn]] ,  alpha' = W'^T W' (y' - m0)            -- O(n^2) per GP.
// One CTA per GP; rows n of the padded L and W (identity rows until now) are overwritten in place.
// =============================================================================================
template <class KC>
__global__ void __launch_bounds__(256) k_append_row(ModelSpec ms, int n_old, double* __restrict__ Lm, double* __restrict__ Wm,
                                                    double* __restrict__ scratch, int* __restrict__ info) {
  const KC kc(ms.kernel);
  __shared__ double red[8];
  __shared__ double s_lnn;
  const int g = blockIdx.x, np = ms.npad, d = ms.d;
  double* Lg = Lm + (size_t)g * np * np;
  double* Wg = Wm + (size_t)g * np * np;
  double* kv = scratch + (size_t)g * 2 * np;     // k_new[0..n_old)
  double* lv = kv + np;                           // l[0..n_old)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double* xnew = ms.Xn + (size_t)n_old * d;
  for (int j = threadIdx.x; j < n_old; j += blockDim.x) {
    double s = 0.0;
    for (int k = 0; k < d; ++k) { const double df = ms.Xn[(size_t)j * d + k] - xnew[k]; s += df * df * ms.inv_ell[g][k]; }
    kv[j] = kc.value(s, ms.sf2[g]);
  }
  __syncthreads();
  double part = 0.0;
  for (int r = warp; r < n_old; r += 8) {          // l_r = sum_{c<=r} W[r][c] k[c]   (one warp per row, coalesced)
    double s = 0.0;
    for (int c = lane; c <= r; c += 32) s += Wg[(size_t)r * np + c] * kv[c];
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
    if (lane == 0) { lv[r] = s; part += s * s; }
  }
  if (lane == 0) red[warp] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    double q = 0.0;
    for (int w = 0; w < 8; ++w) q += red[w];
    const double piv = ms.sf2[g] + ms.sn2[g] - q;
    if (!(piv > 0.0)) { atomicExch(info + g, n_old + 1); s_lnn = 1.0; } else s_lnn = sqrt(piv);
  }
  __syncthreads();
  const double lnn = s_lnn;
  for (int c = threadIdx.x; c < n_old; c += blockDim.x) {     // new rows: L[n][c] = l_c, W[n][c] = -(sum_{r>=c} l_r W[r][c]) / l_nn
    double s = 0.0;
    for (int r = c; r < n_old; ++r) s += lv[r] * Wg[(size_t)r * np + c];
    Lg[(size_t)n_old * np + c] = lv[c];
    Wg[(size_t)n_old * np + c] = -s / lnn;
  }
  if (threadIdx.x == 0) { Lg[(size_t)n_old * np + n_old] = lnn; Wg[(size_t)n_old * np + n_old] = 1.0 / lnn; }
}

int model_append(sbo_ctx* ctx, const double* x_norm_new, const double* y_norm_new) {
  SBO_REQUIRE(ctx->have_model, "sbo_append_sample: no model (call sbo_set_model)");
  SBO_REQUIRE(x_norm_new && y_norm_new, "null pointer");
  ModelSpec& ms = ctx->ms;
  const int n = ms.n, d = ms.d, G = ms.G;
  SBO_REQUIRE(n + 1 <= 16384, "n out of range");
  stage_changed(ctx, Change::APPEND);
  ev_reset(ctx, 0);
  ev_begin(ctx, 0);
  if (n + 1 > ms.npad) {
    // grow the padded factor by one 128-row block: copy L and W into wider matrices, identity on the new diagonal
    const int np0 = ms.npad, np1 = np0 + 128;
    DevBuf nK, nW, nX, nA;
    SBO_TRY(sbo_ensure(ctx, nK, sizeof(double) * (size_t)G * np1 * np1));
    SBO_TRY(sbo_ensure(ctx, nW, sizeof(double) * (size_t)G * np1 * np1));
    SBO_TRY(sbo_ensure(ctx, nX, sizeof(double) * (size_t)np1 * d));
    SBO_TRY(sbo_ensure(ctx, nA, sizeof(double) * (size_t)G * np1 * 2));
    SBO_CUDA(cudaMemsetAsync(nK.p, 0, sizeof(double) * (size_t)G * np1 * np1, ctx->stream));
    SBO_CUDA(cudaMemsetAsync(nW.p, 0, sizeof(double) * (size_t)G * np1 * np1, ctx->stream));
    SBO_CUDA(cudaMemsetAsync(nX.p, 0, sizeof(double) * (size_t)np1 * d, ctx->stream));
    SBO_CUDA(cudaMemcpyAsync(nX.p, ctx->Xn.p, sizeof(double) * (size_t)np0 * d, cudaMemcpyDeviceToDevice, ctx->stream));
    std::vector<double> ones(128, 1.0);
    for (int g = 0; g < G; ++g) {
      for (DevBuf* pr : {&nK, &nW}) {
        const double* src = (const double*)(pr == &nK ? ctx->Kmat.p : ctx->W.p) + (size_t)g * np0 * np0;
        double* dst = (double*)pr->p + (size_t)g * np1 * np1;
        SBO_CUDA(cudaMemcpy2DAsync(dst, sizeof(double) * np1, src, sizeof(double) * np0, sizeof(double) * np0, np0, cudaMemcpyDeviceToDevice, ctx->stream));
        SBO_CUDA(cudaMemcpy2DAsync(dst + (size_t)np0 * np1 + np0, sizeof(double) * (np1 + 1), ones.data(), sizeof(double), sizeof(double), 128,
                                   cudaMemcpyHostToDevice, ctx->stream));
      }
    }
    SBO_CUDA(cudaStreamSynchronize(ctx->stream));
    for (DevBuf* b : {&ctx->Kmat, &ctx->W, &ctx->Xn, &ctx->alpha}) { cudaFree(b->p); }
    ctx->Kmat = nK; ctx->W = nW; ctx->Xn = nX; ctx->alpha = nA;
    ms.npad = np1;
    ms.Xn = (const double*)ctx->Xn.p; ms.alpha = (const double*)ctx->alpha.p; ms.W = (const double*)ctx->W.p;
  }
  const int np = ms.npad;
  // append the inputs (device copies of X_norm / Y_norm grow by one row)
  DevBuf nY;
  SBO_TRY(sbo_ensure(ctx, nY, sizeof(double) * (size_t)(n + 1) * G));
  SBO_CUDA(cudaMemcpyAsync(nY.p, ctx->Yn.p, sizeof(double) * (size_t)n * G, cudaMemcpyDeviceToDevice, ctx->stream));
  SBO_CUDA(cudaMemcpyAsync((double*)nY.p + (size_t)n * G, y_norm_new, sizeof(double) * G, cudaMemcpyHostToDevice, ctx->stream));
  SBO_CUDA(cudaMemcpyAsync((double*)ctx->Xn.p + (size_t)n * d, x_norm_new, sizeof(double) * d, cudaMemcpyHostToDevice, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  cudaFree(ctx->Yn.p);
  ctx->Yn = nY;
  SBO_TRY(sbo_ensure(ctx, ctx->pp_k, sizeof(double) * (size_t)G * 2 * np));
  SBO_CUDA(cudaMemsetAsync(ctx->info.p, 0, sizeof(int) * SBO_MAX_G, ctx->stream));
  with_kernel(ms.kernel, [&](auto kc) {
    k_append_row<decltype(kc)><<<G, 256, 0, ctx->stream>>>(ms, n, (double*)ctx->Kmat.p, (double*)ctx->W.p, (double*)ctx->pp_k.p, (int*)ctx->info.p);
  });
  SBO_LAUNCH_CHECK();
  ms.n = n + 1;
  k_alpha<<<G, 256, 0, ctx->stream>>>(ms, (const double*)ctx->Yn.p, (double*)ctx->alpha.p + (size_t)G * np, (double*)ctx->alpha.p);
  SBO_LAUNCH_CHECK();
  int info[SBO_MAX_G];
  SBO_CUDA(cudaMemcpyAsync(info, ctx->info.p, sizeof(int) * SBO_MAX_G, cudaMemcpyDeviceToHost, ctx->stream));
  ev_end(ctx);
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  ev_collect(ctx);
  for (int g = 0; g < G; ++g)
    if (info[g] != 0) {
      ctx->have_model = false;
      return sbo_fail(ctx, SBO_ERR_NUMERIC, "appended sample makes K of GP " + std::to_string(g) + " numerically singular");
    }
  return SBO_OK;
}

// =============================================================================================
// Batched negative log-likelihood for the hyper-parameter fit (SURVEY.md section 8f row 2).
//   GP.negative_loglikelihood (models/GP_Safe.py:169-192):  K = k(X, X) + (sn2 + 1e-8) I,
//   NLL = y^T K^-1 y + log det K = |L^-1 y|^2 + 2 sum log L_ii   with K = L L^T.
// The reference evaluates it once per DE individual on the host (GP_Safe.py:224); here a whole DE population
// (P hyper-parameter vectors) is factorised in one batch with the blocked-Cholesky kernels above (batch index in the
// place of the GP index).
// =============================================================================================
// hyp[p][0..d) = 1/2 log ell_k, hyp[p][d] = 1/2 log sf2, hyp[p][d+1] = 1/2 log sn2      (GP_Safe.py:180-182)
template <class KC>
__global__ void k_build_K_pop(int kernel, int n, int npad, int d, const double* __restrict__ Xn, const double* __restrict__ hyp,
                              double* __restrict__ K) {
  const KC kc(kernel);
  const int p = blockIdx.z;
  const int r = blockIdx.y * blockDim.y + threadIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= npad || c >= npad) return;
  const double* h = hyp + (size_t)p * (d + 2);
  double v;
  if (r < n && c < n) {
    double s = 0.0;
    for (int k = 0; k < d; ++k) {
      const double df = Xn[r * d + k] - Xn[c * d + k];
      s += df * df / exp(2.0 * h[k]);
    }
    v = kc.value(s, exp(2.0 * h[d]));
    if (r == c) v += exp(2.0 * h[d + 1]) + 1e-8;                       // GP_Safe.py:184
  } else {
    v = (r == c) ? 1.0 : 0.0;
  }
  K[((size_t)p * npad + r) * npad + c] = v;
}

// one CTA per individual: t = L^-1 y by blocked forward substitution, NLL = |t|^2 + 2 sum log L_ii
__global__ void __launch_bounds__(256) k_nll_finish(int n, int npad, const double* __restrict__ Lall, const double* __restrict__ y,
                                                    const int* __restrict__ info, double* __restrict__ nll) {
  extern __shared__ double sh[];        // t[npad] | tmp[NB]
  double* t = sh;
  double* tmp = sh + npad;
  const int p = blockIdx.x;
  const double* L = Lall + (size_t)p * npad * npad;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = 0; i < npad / NB; ++i) {
    const int o = i * NB;
    for (int rr = warp; rr < NB; rr += 8) {           // row o+rr: y_r - sum_{c<o} L[r][c] t[c]
      const int r = o + rr;
      double s = 0.0;
      for (int c = lane; c < o; c += 32) s += L[(size_t)r * npad + c] * t[c];
#pragma unroll
      for (int m = 16; m > 0; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
      if (lane == 0) tmp[rr] = ((r < n) ? y[r] : 0.0) - s;
    }
    __syncthreads();
    if (warp == 0) {                                   // 32x32 diagonal block, lane = row
      double v = tmp[lane];
      for (int j = 0; j < NB; ++j) {
        const double tj = __shfl_sync(0xffffffffu, v, j) / L[(size_t)(o + j) * npad + o + j];
        if (lane == j) v = tj;
        else if (lane > j) v -= L[(size_t)(o + lane) * npad + o + j] * tj;
      }
      t[o + lane] = v;
    }
    __syncthreads();
  }
  double q = 0.0, ld = 0.0;
  for (int r = threadIdx.x; r < n; r += blockDim.x) { q += t[r] * t[r]; ld += log(L[(size_t)r * npad + r]); }
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) { q += __shfl_xor_sync(0xffffffffu, q, m); ld += __shfl_xor_sync(0xffffffffu, ld, m); }
  __syncthreads();
  if (lane == 0) { tmp[warp] = q; tmp[8 + warp] = ld; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double Q = 0.0, LD = 0.0;
    for (int w = 0; w < 8; ++w) { Q += tmp[w]; LD += tmp[8 + w]; }
    nll[p] = (info[p] != 0) ? INFINITY : Q + 2.0 * LD;
  }
}

int nll_batch(sbo_ctx* ctx, int kernel, int n, int d, const double* X_norm, const double* y, int P, const double* hyp, double* nll) {
  SBO_REQUIRE(n >= 1 && n <= 8192, "n out of range");
  SBO_REQUIRE(d >= 1 && d <= SBO_MAX_D, "d out of range (1..8)");
  SBO_REQUIRE(P >= 1 && P <= 65535, "population size out of range (1..65535)");
  SBO_REQUIRE(X_norm && y && hyp && nll, "null pointer");
  SBO_REQUIRE(kernel_valid(kernel), "unknown kernel (SBO_KERNEL_SE, SBO_KERNEL_MATERN32 or SBO_KERNEL_MATERN52)");
  const int np = (int)(cdiv(n, NB) * NB);
  const size_t kbytes = sizeof(double) * (size_t)P * np * np;
  SBO_TRY(sbo_ensure(ctx, ctx->nll_K, kbytes));
  SBO_TRY(sbo_ensure(ctx, ctx->nll_in, sizeof(double) * ((size_t)n * d + n + (size_t)P * (d + 2) + P) + sizeof(int) * (size_t)P));
  double* Xd = (double*)ctx->nll_in.p;
  double* yd = Xd + (size_t)n * d;
  double* hd = yd + n;
  double* od = hd + (size_t)P * (d + 2);
  int* info = (int*)(od + P);
  SBO_CUDA(cudaMemcpyAsync(Xd, X_norm, sizeof(double) * (size_t)n * d, cudaMemcpyHostToDevice, ctx->stream));
  SBO_CUDA(cudaMemcpyAsync(yd, y, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
  SBO_CUDA(cudaMemcpyAsync(hd, hyp, sizeof(double) * (size_t)P * (d + 2), cudaMemcpyHostToDevice, ctx->stream));
  SBO_CUDA(cudaMemsetAsync(info, 0, sizeof(int) * (size_t)P, ctx->stream));
  double* K = (double*)ctx->nll_K.p;
  {
    dim3 b(16, 16), g((unsigned)cdiv(np, 16), (unsigned)cdiv(np, 16), (unsigned)P);
    with_kernel(kernel, [&](auto kc) { k_build_K_pop<decltype(kc)><<<g, b, 0, ctx->stream>>>(kernel, n, np, d, Xd, hd, K); });
    SBO_LAUNCH_CHECK();
  }
  const int nblk = np / NB;
  for (int kb = 0; kb < nblk; ++kb) {
    k_chol_diag<<<P, dim3(NB, NB), 0, ctx->stream>>>(K, np, kb, info);
    SBO_LAUNCH_CHECK();
    const int below = np - (kb + 1) * NB;
    if (below > 0) {
      k_chol_panel<<<dim3((unsigned)cdiv(below, 128), (unsigned)P), 128, 0, ctx->stream>>>(K, np, kb);
      SBO_LAUNCH_CHECK();
      const int nb = below / NB;
      k_chol_update<<<dim3(nb, nb, P), dim3(NB, NB), 0, ctx->stream>>>(K, np, kb);
      SBO_LAUNCH_CHECK();
    }
  }
  SBO_CUDA(cudaFuncSetAttribute(k_nll_finish, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * (8192 + NB))));
  k_nll_finish<<<P, 256, sizeof(double) * (np + NB), ctx->stream>>>(n, np, K, yd, info, od);
  SBO_LAUNCH_CHECK();
  SBO_CUDA(cudaMemcpyAsync(nll, od, sizeof(double) * P, cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}
