// posterior.cu -- GP posterior over the candidate grid (models/GP_Safe.py:310-352 vmapped, as in
// test/test_SafeOpt.py:324-338), trsm form:
//   k_j   = k(s_j),  s_j = sum_k (Xn_jk - xn_k)^2 / ell_k  (SE or Matern)  (K1a, fused ARD cross-covariance)
//   mean  = (m0 + k . alpha) * Ystd + Ymean                                 (K1a epilogue)
//   grad  = d mean / d x (analytic), L_i = max_p ||grad||_inf               (K1c, optional)
//   v     = W k  (W = L^-1 lower triangular),  var = max(0, sf2 - |v|^2) * Ystd^2   (K1b)
//   V rows are optionally kept (FP64 or TF32-rounded FP32) for the fantasy expander GEMM.
// Update after m appended samples (sbo_append_sample leaves rows 0..n0-1 of W unchanged, so v(p)'s first n0 entries stay):
//   e_r = sum_{j<=r} W[r][j] k_j,  r = n0..n0+m-1;   var' = max(0, var/Ystd^2 - sum_r e_r^2) * Ystd^2;   V' = [V ; e]
//   mean and grad from the new alpha                                        (K1a update mode, no solve, no Kx scratch)
#include "common.cuh"
#include <math.h>

#define XC_THREADS 128
#define XC_JT 128
#define XC_MC 8      // update mode: new rows of W per pass (the e_r accumulators live in registers)

__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}


// ---------------------------------------------------------------------------------------------
// Separable SE-ARD factors on a meshgrid.  k(x, X_j) = sf2 * prod_k exp(-1/2 (xn_k - Xn_jk)^2 / ell_k) and on a meshgrid
// xn_k takes only pts_k values, so the cross-covariance of ANY grid point with training point j is a product of d table
// entries  T[g][k][j][i_k]  (sf2 folded into the k = 0 table; rows j >= n are zero).  Tables: G * npad * sum_k pts_k
// doubles (C4: 2 MB, C5: 6 MB) -- L2 resident -- built once per model upload.  With them the N x n cross-covariance
// (GP_Safe.py:146-167 per point in the reference) is never written anywhere: the solve kernel multiplies it into its
// shared-memory stage on the fly (k_solve_fused) and the mean / gradient kernel does the same in registers.
// ---------------------------------------------------------------------------------------------
struct TabSpec {
  const double* base;             // nullptr: no tables (explicit points)
  long long goff;                 // doubles per GP
  long long koff[SBO_MAX_D];      // offset of axis k inside a GP's block
  int pts[SBO_MAX_D];
};
__global__ void __launch_bounds__(256)
k_build_tables(ModelSpec ms, GridSpec gs, TabSpec ts, double* __restrict__ tab) {
  const int k = blockIdx.y, g = blockIdx.z;
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long tot = (long long)ms.npad * ts.pts[k];
  if (e >= tot) return;
  const int j = (int)(e / ts.pts[k]), i = (int)(e % ts.pts[k]);
  double v = 0.0;
  if (j < ms.n) {
    const double xn = (axis_coord(gs, k, i) - ms.Xmean[k]) / ms.Xstd[k];      // GP_Safe.py:326
    const double df = xn - ms.Xn[(size_t)j * ms.d + k];
    v = exp(-0.5 * df * df * ms.inv_ell[g][k]);
    if (k == 0) v *= ms.sf2[g];
  }
  tab[(size_t)g * ts.goff + ts.koff[k] + e] = v;
}

// update mode of K1a (MC > 0): rows r0 .. r0+mr-1 of W in this pass; var is read and rewritten in place; V-row columns
// r0 .. r0+mr-1 are written with the rounding of keep_v = emit (0: none kept)
struct UpdSpec {
  int r0, mr, emit;
  double* var;
  void* vall;
  long long v_count;
};

// ---------------------------------------------------------------------------------------------
// K1a: cross-covariance tile -> Kx scratch [G][npad][P] (points contiguous), mean, optional gradient.
// MC > 0: the update mode -- no Kx; e_r for up to MC new rows of W, staged in shared memory beside X and alpha.
// ---------------------------------------------------------------------------------------------
template <int D, class KC, int MC>
__global__ void __launch_bounds__(XC_THREADS)
k_crosscov(ModelSpec ms, GridSpec gs, long long p0, int P, int valid, double* __restrict__ Kx,
           double* __restrict__ mean_out, long long out_ld, double* __restrict__ gradmax,
           double* __restrict__ grad_out, int grad_gp, TabSpec ts, UpdSpec us) {
  __shared__ double Xs[XC_JT * D];
  __shared__ double As[XC_JT];
  __shared__ double red[XC_THREADS / 32];
  __shared__ double Wr[MC > 0 ? MC * XC_JT : 1];   // referenced only when MC > 0
  const KC kc(ms.kernel);
  const int g = blockIdx.y + ms.g0;
  const int pl = blockIdx.x * XC_THREADS + threadIdx.x;
  const bool in_chunk = pl < P;
  const bool ok = pl < valid;
  double xn[D];
  const double* trow[D];          // table path: &T[g][k][0][i_k] of this point, row stride pts_k
#pragma unroll
  for (int k = 0; k < D; ++k) trow[k] = nullptr;
  if (ok) {
    double x[SBO_MAX_D];
    const long long gp = shard_global(gs, p0 + pl);
    point_coords(gs, gp, x);
#pragma unroll
    for (int k = 0; k < D; ++k) xn[k] = (x[k] - ms.Xmean[k]) / ms.Xstd[k];       // GP_Safe.py:326
    if (ts.base) {
#pragma unroll
      for (int k = 0; k < D; ++k) trow[k] = ts.base + (size_t)(blockIdx.y + ms.g0) * ts.goff + ts.koff[k] + (gp / gs.stride[k]) % gs.pts[k];
    }
  } else {
#pragma unroll
    for (int k = 0; k < D; ++k) xn[k] = 0.0;
  }
  double iell[D];
#pragma unroll
  for (int k = 0; k < D; ++k) iell[k] = ms.inv_ell[g][k];
  const double sf2 = ms.sf2[g];
  const bool want_grad = (gradmax != nullptr) || (grad_out != nullptr && g == grad_gp);
  double acc = 0.0;
  double gk[D];
#pragma unroll
  for (int k = 0; k < D; ++k) gk[k] = 0.0;
  double er[MC > 0 ? MC : 1];
#pragma unroll
  for (int i = 0; i < (MC > 0 ? MC : 1); ++i) er[i] = 0.0;
  double* kcol = Kx + (size_t)g * ms.npad * P + pl;
  for (int j0 = 0; j0 < ms.npad; j0 += XC_JT) {
    __syncthreads();
    for (int e = threadIdx.x; e < XC_JT * D; e += XC_THREADS)
      Xs[e] = (j0 * D + e < ms.npad * D) ? ms.Xn[(size_t)j0 * D + e] : 0.0;
    for (int e = threadIdx.x; e < XC_JT; e += XC_THREADS)
      As[e] = (j0 + e < ms.npad) ? ms.alpha[(size_t)g * ms.npad + j0 + e] : 0.0;
    if constexpr (MC > 0) {
      for (int e = threadIdx.x; e < MC * XC_JT; e += XC_THREADS) {
        const int i = e / XC_JT, c = e % XC_JT;
        Wr[e] = (i < us.mr && j0 + c < ms.n) ? ms.W[((size_t)g * ms.npad + us.r0 + i) * ms.npad + j0 + c] : 0.0;
      }
    }
    __syncthreads();
    const int jn = min(XC_JT, ms.npad - j0);
    if (in_chunk) {
      for (int j = 0; j < jn; ++j) {
        double kv = 0.0;
        if (ok && (j0 + j) < ms.n) {
          double s = 0.0;
          double df[D];
#pragma unroll
          for (int k = 0; k < D; ++k) { df[k] = xn[k] - Xs[j * D + k]; s += df[k] * df[k] * iell[k]; }
          if (ts.base) {                                                         // product of the separable factors
            kv = __ldg(trow[0] + (size_t)(j0 + j) * ts.pts[0]);
#pragma unroll
            for (int k = 1; k < D; ++k) kv *= __ldg(trow[k] + (size_t)(j0 + j) * ts.pts[k]);
          } else {
            kv = kc.value(s, sf2);                                               // GP_Safe.py:165-166
          }
          const double w = As[j] * kv;
          acc += w;
          if (want_grad) {
            const double wg = KC::kIsSE ? w : As[j] * kc.phi(s, sf2);           // dk/dx_k = -phi df_k / ell_k (SE: phi = k)
#pragma unroll
            for (int k = 0; k < D; ++k) gk[k] += wg * df[k];
          }
          if constexpr (MC > 0) {
#pragma unroll
            for (int i = 0; i < MC; ++i) er[i] = fma(Wr[i * XC_JT + j], kv, er[i]);   // rows of W are zero right of the diagonal
          }
        }
        if (Kx) kcol[(size_t)(j0 + j) * P] = kv;
      }
    }
  }
  if (ok && mean_out) mean_out[(size_t)g * out_ld + p0 + pl] = (ms.m0[g] + acc) * ms.Ystd[g] + ms.Ymean[g];   // :342,346
  if (want_grad) {
    double gm = 0.0;
#pragma unroll
    for (int k = 0; k < D; ++k) {
      const double gv = -gk[k] * iell[k] * ms.Ystd[g] / ms.Xstd[k];
      if (ok && grad_out && g == grad_gp) grad_out[(size_t)(p0 + pl) * D + k] = gv;
      gm = fmax(gm, fabs(gv));
    }
    if (gradmax) {
      if (!ok) gm = 0.0;
#pragma unroll
      for (int m = 16; m > 0; m >>= 1) gm = fmax(gm, __shfl_xor_sync(0xffffffffu, gm, m));
      if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = gm;
      __syncthreads();
      if (threadIdx.x == 0) {
        for (int w = 1; w < XC_THREADS / 32; ++w) gm = fmax(gm, red[w]);
        atomicMax((unsigned long long*)(gradmax + g), (unsigned long long)__double_as_longlong(gm));
      }
    }
  }
  if constexpr (MC > 0) {
    if (ok) {
      double s = 0.0;
#pragma unroll
      for (int i = 0; i < MC; ++i) s = fma(er[i], er[i], s);                      // er[i] = 0 for i >= mr
      const size_t o = (size_t)g * out_ld + p0 + pl;
      const double y2 = ms.Ystd[g] * ms.Ystd[g];
      us.var[o] = fmax(0.0, us.var[o] / y2 - s) * y2;                              // a clamped var stays 0
      if (us.emit && g > 0 && us.vall) {                                           // rounding of the solve epilogues
        const int np = ms.npad;
        const size_t row = ((size_t)(g - 1) * us.v_count + p0 + pl) * (us.emit == 3 ? 2 * np : np) + us.r0;
#pragma unroll
        for (int i = 0; i < MC; ++i) {
          if (i >= us.mr) break;
          if (us.emit == 1) {
            reinterpret_cast<double*>(us.vall)[row + i] = er[i];
          } else if (us.emit == 2) {
            reinterpret_cast<float*>(us.vall)[row + i] = to_tf32((float)er[i]);
          } else {
            const float hi = to_tf32((float)er[i]);
            reinterpret_cast<float*>(us.vall)[row + i] = hi;
            reinterpret_cast<float*>(us.vall)[row + i + np] = to_tf32((float)(er[i] - (double)hi));
          }
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// K1b (variant 0, FP64 SIMT): V = W * Kx by 64x64x16 register tiles, triangular in K; the CTA owns
// 64 points and walks all row blocks so |v|^2 is reduced without atomics.
// ---------------------------------------------------------------------------------------------
#define PB_BM 64
#define PB_BP 64
#define PB_BK 16

template <int EMIT>   // 0 none, 1 fp64, 2 fp32 (tf32-rounded), 3 split tf32 pair [hi | lo] (row length 2*npad)
__global__ void __launch_bounds__(256)
k_solve_var(ModelSpec ms, const double* __restrict__ Kx, int P, long long p0, int valid,
            double* __restrict__ var_out, long long out_ld, void* __restrict__ vall, long long v_count) {
  __shared__ double Ws[PB_BK][PB_BM + 1];   // +1: conflict-free transposed stores
  __shared__ __align__(16) double Ks[PB_BK][PB_BP];
  __shared__ double red[16][PB_BP];
  const int g = blockIdx.y + ms.g0;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int np = ms.npad;
  const double* Wg = ms.W + (size_t)g * np * np;
  const double* Kg = Kx + (size_t)g * np * P + (size_t)blockIdx.x * PB_BP;
  double ssum[4] = {0.0, 0.0, 0.0, 0.0};
  const int nrb = np / PB_BM;
  const bool emit = (EMIT != 0) && (g > 0) && (vall != nullptr);
  for (int rb = 0; rb < nrb; ++rb) {
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    const int cmax = (rb + 1) * PB_BM;
    for (int c0 = 0; c0 < cmax; c0 += PB_BK) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int e = tid + 256 * q;
        const int r = e >> 4, c = e & 15;
        Ws[c][r] = Wg[(size_t)(rb * PB_BM + r) * np + c0 + c];
        const int kc = e >> 6, kp = e & 63;
        Ks[kc][kp] = Kg[(size_t)(c0 + kc) * P + kp];
      }
      __syncthreads();
#pragma unroll
      for (int c = 0; c < PB_BK; ++c) {
        const double2 k01 = *reinterpret_cast<const double2*>(&Ks[c][tx * 4]);
        const double2 k23 = *reinterpret_cast<const double2*>(&Ks[c][tx * 4 + 2]);
        const double w[4] = {Ws[c][ty * 4], Ws[c][ty * 4 + 1], Ws[c][ty * 4 + 2], Ws[c][ty * 4 + 3]};
        const double kk[4] = {k01.x, k01.y, k23.x, k23.y};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fma(w[i], kk[j], acc[i][j]);
      }
      __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int i = 0; i < 4; ++i) ssum[j] = fma(acc[i][j], acc[i][j], ssum[j]);
    if (emit) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const long long pl = (long long)blockIdx.x * PB_BP + tx * 4 + j;
        if (pl < valid) {
          const size_t row = ((size_t)(g - 1) * v_count + p0 + pl) * (EMIT == 3 ? 2 * np : np) + rb * PB_BM + ty * 4;
          if (EMIT == 3) {
            float* o = reinterpret_cast<float*>(vall) + row;
            float hi[4], lo[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              hi[i] = to_tf32((float)acc[i][j]);
              lo[i] = to_tf32((float)(acc[i][j] - (double)hi[i]));
            }
            *reinterpret_cast<float4*>(o) = make_float4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<float4*>(o + np) = make_float4(lo[0], lo[1], lo[2], lo[3]);
          } else if (EMIT == 1) {
            double* o = reinterpret_cast<double*>(vall) + row;
            *reinterpret_cast<double2*>(o) = make_double2(acc[0][j], acc[1][j]);
            *reinterpret_cast<double2*>(o + 2) = make_double2(acc[2][j], acc[3][j]);
          } else {
            float* o = reinterpret_cast<float*>(vall) + row;
            *reinterpret_cast<float4*>(o) = make_float4(to_tf32((float)acc[0][j]), to_tf32((float)acc[1][j]),
                                                        to_tf32((float)acc[2][j]), to_tf32((float)acc[3][j]));
          }
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) red[ty][tx * 4 + j] = ssum[j];
  __syncthreads();
  if (tid < PB_BP) {
    double s = 0.0;
#pragma unroll
    for (int t = 0; t < 16; ++t) s += red[t][tid];
    const long long pl = (long long)blockIdx.x * PB_BP + tid;
    if (pl < valid) {
      const double v = fmax(0.0, ms.sf2[g] - s);                                  // GP_Safe.py:343
      var_out[(size_t)g * out_ld + p0 + pl] = v * ms.Ystd[g] * ms.Ystd[g];        // :347
    }
  }
}

// ---------------------------------------------------------------------------------------------
// K1b (variant 1, FP64 tensor cores): the same V = W * Kx with mma.sync.m8n8k4.f64 (DMMA; sm_100a has no FP64
// tcgen05 path).  CTA = 128 rows x 64 points per row block, 8 warps of 32x32, cp.async double-buffered K chunks of
// 32; strides 36 / 72 doubles make the fragment loads conflict-free.  The CTA walks all row blocks so |v|^2 needs
// no atomics; triangular in K as above.
// ---------------------------------------------------------------------------------------------
#define DV_BM 128
#define DV_BP 64
#define DV_BK 32
#define DV_WS 36   // Ws row stride (doubles): 36 = 4 mod 16
#define DV_KS 72   // Ks row stride (doubles): 72 = 8 mod 16
#define DV_STAGE (DV_BM * DV_WS + DV_BK * DV_KS)
#define DV_SMEM (2 * DV_STAGE * 8 + 4 * DV_BP * 8)
#define DV_SMEM_F (DV_SMEM + SBO_MAX_D * DV_BP * 4)   // fused kernel: + per-point table offsets

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}


// one K chunk of the DMMA solve for fragments I0..3 of the warp (fragment i = rows i*32 + wr*8 .. +7 of the row block)
template <int I0>
__device__ __forceinline__ void dv_chunk(double (&acc)[4][4][2], const double* __restrict__ Ws, const double* __restrict__ Ks,
                                         int wr, int wp, int grp, int tig) {
#pragma unroll
  for (int k0 = 0; k0 < DV_BK; k0 += 4) {
    double a[4], b[4];
#pragma unroll
    for (int i = I0; i < 4; ++i) a[i] = Ws[(i * 32 + wr * 8 + grp) * DV_WS + k0 + tig];
#pragma unroll
    for (int j = 0; j < 4; ++j) b[j] = Ks[(k0 + tig) * DV_KS + wp * 32 + j * 8 + grp];
#pragma unroll
    for (int i = I0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
  }
}

template <int EMIT>
__global__ void __launch_bounds__(256, 2)
k_solve_var_dmma(ModelSpec ms, const double* __restrict__ Kx, int P, long long p0, int valid,
                 double* __restrict__ var_out, long long out_ld, void* __restrict__ vall, long long v_count) {
  extern __shared__ __align__(16) double dsm[];
  double* red = dsm + 2 * DV_STAGE;                 // [4][DV_BP]
  const int g = blockIdx.y + ms.g0;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int grp = lane >> 2, tig = lane & 3;
  const int wr = warp & 3, wp = warp >> 2;          // warp tile: rows wr*32.., points wp*32..
  const int np = ms.npad;
  const double* Wg = ms.W + (size_t)g * np * np;
  const double* Kg = Kx + (size_t)g * np * P + (size_t)blockIdx.x * DV_BP;
  const bool emit = (EMIT != 0) && (g > 0) && (vall != nullptr);
  double ssum[4][2];
#pragma unroll
  for (int j = 0; j < 4; ++j) ssum[j][0] = ssum[j][1] = 0.0;

  auto load_chunk = [&](int stage, int rb, int c0) {
    double* Ws = dsm + stage * DV_STAGE;
    double* Ks = Ws + DV_BM * DV_WS;
#pragma unroll
    for (int q = 0; q < 8; ++q) {                   // W tile: 128 rows x 32 cols = 2048 x 16 B
      const int e = tid + 256 * q;
      const int r = e >> 4, c2 = (e & 15) * 2;
      cp_async16(Ws + r * DV_WS + c2, Wg + (size_t)(rb * DV_BM + r) * np + c0 + c2);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {                   // Kx tile: 32 rows x 64 points = 1024 x 16 B
      const int e = tid + 256 * q;
      const int r = e >> 5, c2 = (e & 31) * 2;
      cp_async16(Ks + r * DV_KS + c2, Kg + (size_t)(c0 + r) * P + c2);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  const int nrb = np / DV_BM;
  int it = 0;                                       // chunk counter over ALL row blocks: the ring never drains between them
  load_chunk(0, 0, 0);
  for (int rb = 0; rb < nrb; ++rb) {
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    const int nk = (rb + 1) * DV_BM / DV_BK;
    for (int kc = 0; kc < nk; ++kc, ++it) {
      // prefetch the successor chunk -- the first chunk of the NEXT row block after the last one of this block, so that
      // it lands while this block's epilogue (|v|^2, V rows) runs
      const bool last = kc + 1 == nk;
      if (!last || rb + 1 < nrb) {
        load_chunk((it + 1) & 1, last ? rb + 1 : rb, last ? 0 : (kc + 1) * DV_BK);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
      } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
      __syncthreads();
      const double* Ws = dsm + (it & 1) * DV_STAGE;
      const double* Ks = Ws + DV_BM * DV_WS;
      // W is lower triangular: rows of quarter i (32 rows) of the block need columns <= rb*128 + i*32 + 31 only, i.e. K
      // chunks kc <= rb*4 + i.  Every warp owns 8 rows of EACH quarter (fragment i = rows i*32 + wr*8 .. +7), so in the
      // diagonal block all warps skip the same zero fragments: 10 fragment-chunks each instead of 4/8/12/16 per warp.
      const int iq = kc - rb * (DV_BM / DV_BK);        // quarter index of this chunk inside the diagonal block (<= 0 before it)
      // real (warp-uniform) branches over compile-time fragment ranges: a predicated-off DMMA still occupies the FP64
      // tensor pipe (measured: ptxas predicates `if (i >= iq)`, and the kernel time does not move)
      if (iq <= 0) dv_chunk<0>(acc, Ws, Ks, wr, wp, grp, tig);
      else if (iq == 1) dv_chunk<1>(acc, Ws, Ks, wr, wp, grp, tig);
      else if (iq == 2) dv_chunk<2>(acc, Ws, Ks, wr, wp, grp, tig);
      else dv_chunk<3>(acc, Ws, Ks, wr, wp, grp, tig);
      __syncthreads();
    }
    // row-block epilogue: acc[i][j][e] = v[row = rb*128 + i*32 + wr*8 + grp][point = wp*32 + j*8 + 2*tig + e]
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
#pragma unroll
        for (int i = 0; i < 4; ++i) ssum[j][e] = fma(acc[i][j][e], acc[i][j][e], ssum[j][e]);
        if (emit) {
          const long long pl = (long long)blockIdx.x * DV_BP + wp * 32 + j * 8 + 2 * tig + e;
          if (pl < valid) {
            const size_t rowbase = ((size_t)(g - 1) * v_count + p0 + pl) * (EMIT == 3 ? 2 * np : np) + rb * DV_BM + wr * 8 + grp;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const double v = acc[i][j][e];
              if (EMIT == 1) {
                reinterpret_cast<double*>(vall)[rowbase + i * 32] = v;
              } else if (EMIT == 2) {
                reinterpret_cast<float*>(vall)[rowbase + i * 32] = to_tf32((float)v);
              } else {
                const float hi = to_tf32((float)v);
                reinterpret_cast<float*>(vall)[rowbase + i * 32] = hi;
                reinterpret_cast<float*>(vall)[rowbase + i * 32 + np] = to_tf32((float)(v - (double)hi));
              }
            }
          }
        }
      }
  }
  // reduce |v|^2 over the 8 lanes that share a point (same tig, all grp) and over the 4 row warps
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      double s = ssum[j][e];
      s += __shfl_xor_sync(0xffffffffu, s, 4);
      s += __shfl_xor_sync(0xffffffffu, s, 8);
      s += __shfl_xor_sync(0xffffffffu, s, 16);
      if (grp == 0) red[wr * DV_BP + wp * 32 + j * 8 + 2 * tig + e] = s;
    }
  __syncthreads();
  if (tid < DV_BP) {
    const double s = red[tid] + red[DV_BP + tid] + red[2 * DV_BP + tid] + red[3 * DV_BP + tid];
    const long long pl = (long long)blockIdx.x * DV_BP + tid;
    if (pl < valid) {
      const double v = fmax(0.0, ms.sf2[g] - s);                                  // GP_Safe.py:343
      var_out[(size_t)g * out_ld + p0 + pl] = v * ms.Ystd[g] * ms.Ystd[g];        // :347
    }
  }
}

// K1 fused (meshgrid): the same kernel, but the cross-covariance chunk Ks[32 training rows][64 points] is not read from a
// scratch matrix: every thread multiplies the separable table factors of its 2 points x 4 rows straight into the
// shared-memory stage (TabSpec).  No N x n matrix exists anywhere; DRAM traffic is the outputs plus the L2-resident
// tables.  EMIT is a run-time argument here (it only steers the per-row-block epilogue).
template <int D>
__global__ void __launch_bounds__(256, 2)
k_solve_fused(ModelSpec ms, GridSpec gs, TabSpec ts, int EMIT, long long p0, int valid,
              double* __restrict__ var_out, long long out_ld, void* __restrict__ vall, long long v_count) {
  extern __shared__ __align__(16) double dsm[];
  double* red = dsm + 2 * DV_STAGE;                 // [4][DV_BP]
  const int g = blockIdx.y + ms.g0;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int grp = lane >> 2, tig = lane & 3;
  const int wr = warp & 3, wp = warp >> 2;          // warp tile: rows wr*32.., points wp*32..
  const int np = ms.npad;
  const double* Wg = ms.W + (size_t)g * np * np;
  // table entry of point p of this CTA for training row j and axis k: tg[pidx[k][p] + j * pts_k]; the 32-bit offsets
  // live in shared memory (the kernel has no registers to spare: 64 accumulators + fragments at 2 CTAs per SM)
  const double* tg = ts.base + (size_t)g * ts.goff;
  int* pidx = reinterpret_cast<int*>(red + 4 * DV_BP);          // [D][DV_BP]
  for (int e = tid; e < D * DV_BP; e += 256) {
    const int k = e / DV_BP, p = e - k * DV_BP;
    const long long pl = (long long)blockIdx.x * DV_BP + p;
    const long long gp = shard_global(gs, p0 + (pl < valid ? pl : 0));
    pidx[e] = (int)(ts.koff[k] + (gp / gs.stride[k]) % gs.pts[k]);
  }
  __syncthreads();
  const bool emit = (EMIT != 0) && (g > 0) && (vall != nullptr);
  double ssum[4][2];
#pragma unroll
  for (int j = 0; j < 4; ++j) ssum[j][0] = ssum[j][1] = 0.0;

  auto load_chunk = [&](int stage, int rb, int c0) {
    double* Ws = dsm + stage * DV_STAGE;
    double* Ks = Ws + DV_BM * DV_WS;
#pragma unroll
    for (int q = 0; q < 8; ++q) {                   // W tile: 128 rows x 32 cols = 2048 x 16 B
      const int e = tid + 256 * q;
      const int r = e >> 4, c2 = (e & 15) * 2;
      cp_async16(Ws + r * DV_WS + c2, Wg + (size_t)(rb * DV_BM + r) * np + c0 + c2);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
#pragma unroll
    for (int q = 0; q < 4; ++q) {                   // cross-covariance tile: 32 training rows x 64 points, generated
      const int r = warp + 8 * q;                   // (tid + 256 q) >> 5
      const int j = c0 + r;
      int2 o = *reinterpret_cast<const int2*>(pidx + 2 * lane);
      double va = __ldg(tg + o.x + j * ts.pts[0]), vb = __ldg(tg + o.y + j * ts.pts[0]);
#pragma unroll
      for (int k = 1; k < D; ++k) {
        o = *reinterpret_cast<const int2*>(pidx + k * DV_BP + 2 * lane);
        va *= __ldg(tg + o.x + j * ts.pts[k]); vb *= __ldg(tg + o.y + j * ts.pts[k]);
      }
      *reinterpret_cast<double2*>(Ks + r * DV_KS + 2 * lane) = make_double2(va, vb);
    }
  };

  const int nrb = np / DV_BM;
  for (int rb = 0; rb < nrb; ++rb) {
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    const int nk = (rb + 1) * DV_BM / DV_BK;
    load_chunk(0, rb, 0);
    for (int kc = 0; kc < nk; ++kc) {
      if (kc + 1 < nk) {
        load_chunk((kc + 1) & 1, rb, (kc + 1) * DV_BK);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
      } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
      __syncthreads();
      const double* Ws = dsm + (kc & 1) * DV_STAGE;
      const double* Ks = Ws + DV_BM * DV_WS;
      // W is lower triangular: rows of quarter i (32 rows) of the block need columns <= rb*128 + i*32 + 31 only, i.e. K
      // chunks kc <= rb*4 + i.  Every warp owns 8 rows of EACH quarter (fragment i = rows i*32 + wr*8 .. +7), so in the
      // diagonal block all warps skip the same zero fragments: 10 fragment-chunks each instead of 4/8/12/16 per warp.
      const int iq = kc - rb * (DV_BM / DV_BK);        // quarter index of this chunk inside the diagonal block (<= 0 before it)
      // real (warp-uniform) branches over compile-time fragment ranges: a predicated-off DMMA still occupies the FP64
      // tensor pipe (measured: ptxas predicates `if (i >= iq)`, and the kernel time does not move)
      if (iq <= 0) dv_chunk<0>(acc, Ws, Ks, wr, wp, grp, tig);
      else if (iq == 1) dv_chunk<1>(acc, Ws, Ks, wr, wp, grp, tig);
      else if (iq == 2) dv_chunk<2>(acc, Ws, Ks, wr, wp, grp, tig);
      else dv_chunk<3>(acc, Ws, Ks, wr, wp, grp, tig);
      __syncthreads();
    }
    // row-block epilogue: acc[i][j][e] = v[row = rb*128 + i*32 + wr*8 + grp][point = wp*32 + j*8 + 2*tig + e]
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
#pragma unroll
        for (int i = 0; i < 4; ++i) ssum[j][e] = fma(acc[i][j][e], acc[i][j][e], ssum[j][e]);
        if (emit) {
          const long long pl = (long long)blockIdx.x * DV_BP + wp * 32 + j * 8 + 2 * tig + e;
          if (pl < valid) {
            const size_t rowbase = ((size_t)(g - 1) * v_count + p0 + pl) * (EMIT == 3 ? 2 * np : np) + rb * DV_BM + wr * 8 + grp;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const double v = acc[i][j][e];
              if (EMIT == 1) {
                reinterpret_cast<double*>(vall)[rowbase + i * 32] = v;
              } else if (EMIT == 2) {
                reinterpret_cast<float*>(vall)[rowbase + i * 32] = to_tf32((float)v);
              } else {
                const float hi = to_tf32((float)v);
                reinterpret_cast<float*>(vall)[rowbase + i * 32] = hi;
                reinterpret_cast<float*>(vall)[rowbase + i * 32 + np] = to_tf32((float)(v - (double)hi));
              }
            }
          }
        }
      }
  }
  // reduce |v|^2 over the 8 lanes that share a point (same tig, all grp) and over the 4 row warps
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      double s = ssum[j][e];
      s += __shfl_xor_sync(0xffffffffu, s, 4);
      s += __shfl_xor_sync(0xffffffffu, s, 8);
      s += __shfl_xor_sync(0xffffffffu, s, 16);
      if (grp == 0) red[wr * DV_BP + wp * 32 + j * 8 + 2 * tig + e] = s;
    }
  __syncthreads();
  if (tid < DV_BP) {
    const double s = red[tid] + red[DV_BP + tid] + red[2 * DV_BP + tid] + red[3 * DV_BP + tid];
    const long long pl = (long long)blockIdx.x * DV_BP + tid;
    if (pl < valid) {
      const double v = fmax(0.0, ms.sf2[g] - s);                                  // GP_Safe.py:343
      var_out[(size_t)g * out_ld + p0 + pl] = v * ms.Ystd[g] * ms.Ystd[g];        // :347
    }
  }
}

// ---------------------------------------------------------------------------------------------
// host drivers
// ---------------------------------------------------------------------------------------------
static int crosscov_dispatch(sbo_ctx* ctx, const GridSpec& gs, long long p0, int P, int valid, double* Kx,
                             double* mean_out, long long out_ld, double* gradmax, double* grad_out, int grad_gp,
                             const TabSpec& ts = TabSpec{}) {
  const int g0 = ctx->post_g0;
  ModelSpec msl = ctx->ms; msl.g0 = g0;
  dim3 grid((unsigned)cdiv(P, XC_THREADS), (unsigned)(ctx->ms.G - g0));
  with_int<1, SBO_MAX_D>(msl.d, [&](auto D) { with_kernel(msl.kernel, [&](auto kc) {
    k_crosscov<D, decltype(kc), 0><<<grid, XC_THREADS, 0, ctx->stream>>>(msl, gs, p0, P, valid, Kx, mean_out, out_ld, gradmax,
                                                                         grad_out, grad_gp, ts, UpdSpec{});
  }); });
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

static int solve_dispatch(sbo_ctx* ctx, const double* Kx, int P, long long p0, int valid, double* var_out,
                          long long out_ld, int keep_v, void* vall, long long v_count) {
  const int g0 = ctx->post_g0;
  ModelSpec msl = ctx->ms; msl.g0 = g0;
  SBO_TRY((with_int<0, 3>(keep_v, [&](auto EMIT) -> int {
    void* v = EMIT ? vall : nullptr;
    const long long vc = EMIT ? v_count : 0;
    if (ctx->opt_posterior_variant == 1) {   // FP64 tensor-core (DMMA) kernel
      dim3 grid((unsigned)(P / DV_BP), (unsigned)(ctx->ms.G - g0));
      // the attribute is per device and a process may hold contexts on several GPUs: set it before every launch
      SBO_CUDA(cudaFuncSetAttribute(k_solve_var_dmma<EMIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, DV_SMEM));
      k_solve_var_dmma<EMIT><<<grid, 256, DV_SMEM, ctx->stream>>>(msl, Kx, P, p0, valid, var_out, out_ld, v, vc);
    } else {
      dim3 grid((unsigned)(P / PB_BP), (unsigned)(ctx->ms.G - g0));
      k_solve_var<EMIT><<<grid, 256, 0, ctx->stream>>>(msl, Kx, P, p0, valid, var_out, out_ld, v, vc);
    }
    return SBO_OK;
  })));
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

// K1 fused path (meshgrid grids, option "posterior_fused", default 0): separable factor tables, table-based mean /
// gradient kernel (no Kx store), fused solve kernel (no Kx load).
static int build_tables(sbo_ctx* ctx, TabSpec* ts) {
  const ModelSpec& ms = ctx->ms;
  const GridSpec& gs = ctx->gs;
  *ts = TabSpec{};
  long long tot = 0;
  for (int k = 0; k < gs.d; ++k) { ts->koff[k] = tot; ts->pts[k] = (int)gs.pts[k]; tot += (long long)ms.npad * gs.pts[k]; }
  ts->goff = tot;
  SBO_TRY(sbo_ensure(ctx, ctx->tabs, sizeof(double) * (size_t)tot * ms.G));
  ts->base = (const double*)ctx->tabs.p;
  long long mx = 0;
  for (int k = 0; k < gs.d; ++k) mx = mx > (long long)ms.npad * gs.pts[k] ? mx : (long long)ms.npad * gs.pts[k];
  k_build_tables<<<dim3((unsigned)cdiv(mx, 256), gs.d, ms.G), 256, 0, ctx->stream>>>(ms, gs, *ts, (double*)ctx->tabs.p);
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

static int fused_dispatch(sbo_ctx* ctx, const TabSpec& ts, int emit, long long p0, int P, int valid, double* var_out, long long out_ld,
                          void* vall, long long v_count) {
  dim3 grid((unsigned)(P / DV_BP), (unsigned)ctx->ms.G);
  SBO_TRY((with_int<1, SBO_MAX_D>(ctx->ms.d, [&](auto D) -> int {
    SBO_CUDA(cudaFuncSetAttribute(k_solve_fused<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, DV_SMEM_F));
    k_solve_fused<D><<<grid, 256, DV_SMEM_F, ctx->stream>>>(ctx->ms, ctx->gs, ts, emit, p0, valid, var_out, out_ld, vall, v_count);
    return SBO_OK;
  })));
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

// Points per chunk.  The cross-covariance tile Kx[G][npad][P] is produced by k_crosscov and consumed by the solve kernel
// of the same chunk (option "posterior_chunk_mb", default 1024).  Measured at C4 (profiles/r02_posterior_chunk_ab.txt):
// L2-resident chunks (24-96 MB) avoid the HBM round trip of the tile but cost more than they save -- 11-18 launches
// of partial waves instead of one: crosscov 8.3 -> 28 ms, solve 40 -> 44 ms -- so the large chunk stays the default.
// Never fewer points than one full wave of the solve kernel needs (2 CTAs of 64 points per SM and GP).
static long long chunk_points(const sbo_ctx* ctx, const ModelSpec& ms, long long count) {
  const size_t per_pt = (size_t)ms.G * ms.npad * sizeof(double);
  const long long mb = ctx->opt_posterior_chunk_mb > 0 ? ctx->opt_posterior_chunk_mb : 1024;
  long long p = (long long)((size_t)mb << 20) / (long long)per_pt;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  const long long wave = (long long)cdiv((long long)sms * 2, ms.G) * 64;     // points that fill one wave of the solve kernel
  if (p < wave) p = wave;
  p = (p / 128) * 128;
  if (p < 128) p = 128;
  const long long need = cdiv(count, 128) * 128;
  return p < need ? p : need;
}

int posterior_run(sbo_ctx* ctx, int with_grad, int keep_v) {
  SBO_REQUIRE(ctx->have_model, "sbo_posterior: no model (call sbo_set_model)");
  SBO_REQUIRE(ctx->have_grid, "sbo_posterior: no grid (call sbo_set_grid / sbo_set_points)");
  SBO_REQUIRE(ctx->gs.d == ctx->ms.d, "grid and model dimensions differ");
  SBO_REQUIRE(keep_v >= 0 && keep_v <= 3, "keep_v must be 0, 1, 2 or 3");
  stage_changed(ctx, Change::POSTERIOR);
  const ModelSpec& ms = ctx->ms;
  const long long count = ctx->gs.count;
  SBO_REQUIRE(count > 0, "empty shard");
  SBO_TRY(sbo_ensure(ctx, ctx->mean, sizeof(double) * (size_t)ms.G * count));
  SBO_TRY(sbo_ensure(ctx, ctx->var, sizeof(double) * (size_t)ms.G * count));
  SBO_TRY(sbo_ensure(ctx, ctx->lmax, sizeof(double) * SBO_MAX_G));
  // meshgrid + DMMA variant: fused path, no cross-covariance scratch at all (one "chunk" = the whole shard)
  // the separable factor tables exist for the SE kernel only: a Matern model ignores "posterior_fused" / "posterior_tables"
  const bool separable = ctx->gs.kind == 1 && ms.kernel == SBO_KERNEL_SE;
  const bool fused = separable && ctx->opt_posterior_variant == 1 && ctx->opt_posterior_fused;
  const long long P = fused ? cdiv(count, 128) * 128 : chunk_points(ctx, ms, count);
  if (!fused) SBO_TRY(sbo_ensure(ctx, ctx->kx, sizeof(double) * (size_t)ms.G * ms.npad * P));
  if (keep_v && ms.G > 1) {
    const size_t esz = keep_v == 1 ? sizeof(double) : (keep_v == 3 ? 2 * sizeof(float) : sizeof(float));
    SBO_TRY(sbo_ensure(ctx, ctx->vall, esz * (size_t)(ms.G - 1) * count * ms.npad));
  }
  SBO_CUDA(cudaMemsetAsync(ctx->lmax.p, 0, sizeof(double) * SBO_MAX_G, ctx->stream));
  ev_reset(ctx, 1); ev_reset(ctx, 2);
  // meshgrids: the cross-covariance kernel takes its kernel values from the separable factor tables (d loads + d-1
  // multiplies instead of an FP64 exp per entry) whether or not the solve is fused
  TabSpec ts{};
  if (separable && (fused || ctx->opt_posterior_tables)) {
    ev_begin(ctx, 1);
    SBO_TRY(build_tables(ctx, &ts));
    ev_end(ctx);
  }
  for (long long p0 = 0; p0 < count; p0 += P) {
    const int valid = (int)((count - p0) < P ? (count - p0) : P);
    const int Pc = (int)P;
    ev_begin(ctx, 1);
    SBO_TRY(crosscov_dispatch(ctx, ctx->gs, p0, Pc, valid, fused ? nullptr : (double*)ctx->kx.p, (double*)ctx->mean.p, count,
                              with_grad ? (double*)ctx->lmax.p : nullptr, nullptr, -1, ts));
    ev_end(ctx);
    ev_begin(ctx, 2);
    if (fused)
      SBO_TRY(fused_dispatch(ctx, ts, (ms.G > 1) ? keep_v : 0, p0, Pc, valid, (double*)ctx->var.p, count, ctx->vall.p, count));
    else
      SBO_TRY(solve_dispatch(ctx, (const double*)ctx->kx.p, Pc, p0, valid, (double*)ctx->var.p, count,
                             (ms.G > 1) ? keep_v : 0, ctx->vall.p, count));
    ev_end(ctx);
  }
  ctx->up.n = ms.n; ctx->up.npad = ms.npad;
  ctx->up.with_grad = with_grad != 0; ctx->up.keep_v = keep_v;
  stage_changed(ctx, Change::POSTERIOR_DONE);
  return SBO_OK;
}

// sbo_posterior_update: the last posterior_run brought up to the model after the sbo_append_sample calls since.  Rows
// up.n .. n-1 of W are the new ones; ceil(m / XC_MC) passes of the K1a update mode, the first also writes mean and the
// Lipschitz constants (bitwise what posterior_run computes with the default options: the same loop in the same order).
int posterior_update(sbo_ctx* ctx, sbo_update_info* info) {
  SBO_REQUIRE(ctx->have_model, "sbo_posterior_update: no model");
  SBO_REQUIRE(ctx->up.valid, "sbo_posterior_update: no posterior to update -- none since the last sbo_set_model, sbo_set_grid, "
                             "sbo_set_points or sbo_set_shard, or its V rows were released (call sbo_posterior)");
  const ModelSpec& ms = ctx->ms;
  const int m = ms.n - ctx->up.n;
  info->rows = m; info->recomputed = 0; info->pad = 0;
  if (m == 0) return SBO_OK;
  ev_reset(ctx, 8);
  if (ctx->keep_v && ms.npad != ctx->up.npad) {    // the V-row stride changed with the padding: recompute
    SBO_TRY(posterior_run(ctx, ctx->up.with_grad, ctx->up.keep_v));
    info->recomputed = 1;
    return SBO_OK;
  }
  const long long count = ctx->gs.count;
  const bool with_grad = ctx->up.with_grad;
  if (with_grad) SBO_CUDA(cudaMemsetAsync(ctx->lmax.p, 0, sizeof(double) * SBO_MAX_G, ctx->stream));
  const long long CH = 1LL << 30;                  // points per launch (int offsets inside the kernel)
  for (long long p0 = 0; p0 < count; p0 += CH) {
    const int valid = (int)((count - p0) < CH ? (count - p0) : CH);
    for (int r0 = ctx->up.n; r0 < ms.n; r0 += XC_MC) {
      const bool first = r0 == ctx->up.n;
      UpdSpec us{r0, (ms.n - r0) < XC_MC ? (ms.n - r0) : XC_MC, ctx->keep_v, (double*)ctx->var.p, ctx->vall.p, count};
      dim3 grid((unsigned)cdiv(valid, XC_THREADS), (unsigned)ms.G);
      ev_begin(ctx, 8);
      with_int<1, SBO_MAX_D>(ms.d, [&](auto D) { with_kernel(ms.kernel, [&](auto kc) {
        k_crosscov<D, decltype(kc), XC_MC><<<grid, XC_THREADS, 0, ctx->stream>>>(
            ms, ctx->gs, p0, valid, valid, nullptr, first ? (double*)ctx->mean.p : nullptr, count,
            (first && with_grad) ? (double*)ctx->lmax.p : nullptr, nullptr, -1, TabSpec{}, us);
      }); });
      ev_end(ctx);
      SBO_LAUNCH_CHECK();
    }
  }
  ctx->up.n = ms.n; ctx->up.npad = ms.npad;
  stage_changed(ctx, Change::POSTERIOR_DONE);
  return SBO_OK;
}

// GP_inference at arbitrary points (GP_Safe.py:310-352), used by BO.mean/ucb/lcb (SafeOpt.py:29-45)
static int points_common(sbo_ctx* ctx, int64_t m, const double* x, GridSpec& tmp, DevBuf& xbuf) {
  SBO_REQUIRE(ctx->have_model, "no model (call sbo_set_model)");
  SBO_REQUIRE(m >= 1 && x, "bad points");
  SBO_TRY(sbo_ensure(ctx, xbuf, sizeof(double) * (size_t)m * ctx->ms.d));
  SBO_CUDA(cudaMemcpyAsync(xbuf.p, x, sizeof(double) * (size_t)m * ctx->ms.d, cudaMemcpyHostToDevice, ctx->stream));
  tmp = GridSpec{};
  tmp.kind = 2; tmp.d = ctx->ms.d; tmp.N = m; tmp.first = 0; tmp.count = m;
  tmp.explicit_pts = (const double*)xbuf.p;
  return SBO_OK;
}

int posterior_points(sbo_ctx* ctx, int64_t m, const double* x, double* mean, double* var) {
  GridSpec tmp;
  DevBuf &xbuf = ctx->pp_x, &mbuf = ctx->pp_m, &vbuf = ctx->pp_v, &kbuf = ctx->pp_k;
  SBO_TRY(points_common(ctx, m, x, tmp, xbuf));
  const ModelSpec& ms = ctx->ms;
  SBO_TRY(sbo_ensure(ctx, mbuf, sizeof(double) * (size_t)ms.G * m));
  SBO_TRY(sbo_ensure(ctx, vbuf, sizeof(double) * (size_t)ms.G * m));
  const long long P = chunk_points(ctx, ms, m);
  SBO_TRY(sbo_ensure(ctx, kbuf, sizeof(double) * (size_t)ms.G * ms.npad * P));
  for (long long p0 = 0; p0 < m; p0 += P) {
    const int valid = (int)((m - p0) < P ? (m - p0) : P);
    SBO_TRY(crosscov_dispatch(ctx, tmp, p0, (int)P, valid, (double*)kbuf.p, (double*)mbuf.p, m, nullptr, nullptr, -1));
    SBO_TRY(solve_dispatch(ctx, (const double*)kbuf.p, (int)P, p0, valid, (double*)vbuf.p, m, 0, nullptr, 0));
  }
  std::vector<double> hm((size_t)ms.G * m), hv((size_t)ms.G * m);
  SBO_CUDA(cudaMemcpyAsync(hm.data(), mbuf.p, sizeof(double) * hm.size(), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaMemcpyAsync(hv.data(), vbuf.p, sizeof(double) * hv.size(), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int64_t p = 0; p < m; ++p)
    for (int g = 0; g < ms.G; ++g) {
      if (mean) mean[p * ms.G + g] = hm[(size_t)g * m + p];
      if (var) var[p * ms.G + g] = hv[(size_t)g * m + p];
    }
  return SBO_OK;
}

// device scratch posterior_vrows_dev allocates for m points: pp_m and pp_v (mv_bytes each) and pp_k (k_bytes)
void posterior_vrows_scratch(const sbo_ctx* ctx, long long m, size_t* mv_bytes, size_t* k_bytes) {
  const ModelSpec& ms = ctx->ms;
  *mv_bytes = sizeof(double) * (size_t)ms.G * m;
  *k_bytes = sizeof(double) * (size_t)ms.G * ms.npad * chunk_points(ctx, ms, m);
}

// FP64 rows V_i = L_i^-1 K_i(X, p) of m explicit points already on the device (raw coordinates, [m][d] row-major), for
// the constraints: vout[(G-1)][m][npad].  Used by the FP64 re-evaluation of the split-TF32 fantasy expander.
int posterior_vrows_dev(sbo_ctx* ctx, long long m, const double* pts_dev, double* vout) {
  SBO_REQUIRE(ctx->have_model && m >= 1 && pts_dev && vout, "posterior_vrows_dev: bad arguments");
  const ModelSpec& ms = ctx->ms;
  GridSpec tmp{};
  tmp.kind = 2; tmp.d = ms.d; tmp.N = m; tmp.first = 0; tmp.count = m;
  tmp.explicit_pts = pts_dev;
  SBO_TRY(sbo_ensure(ctx, ctx->pp_m, sizeof(double) * (size_t)ms.G * m));
  SBO_TRY(sbo_ensure(ctx, ctx->pp_v, sizeof(double) * (size_t)ms.G * m));
  const long long P = chunk_points(ctx, ms, m);
  SBO_TRY(sbo_ensure(ctx, ctx->pp_k, sizeof(double) * (size_t)ms.G * ms.npad * P));
  ctx->post_g0 = ms.G > 1 ? 1 : 0;               // the objective GP's rows are not needed
  int rc = SBO_OK;
  for (long long p0 = 0; p0 < m && rc == SBO_OK; p0 += P) {
    const int valid = (int)((m - p0) < P ? (m - p0) : P);
    rc = crosscov_dispatch(ctx, tmp, p0, (int)P, valid, (double*)ctx->pp_k.p, (double*)ctx->pp_m.p, m, nullptr, nullptr, -1);
    if (rc == SBO_OK) rc = solve_dispatch(ctx, (const double*)ctx->pp_k.p, (int)P, p0, valid, (double*)ctx->pp_v.p, m, 1, vout, m);
  }
  ctx->post_g0 = 0;
  return rc;
}

int posterior_point_grad(sbo_ctx* ctx, int gp, int64_t m, const double* x, double* grad) {
  GridSpec tmp;
  DevBuf &xbuf = ctx->pp_x, &gbuf = ctx->pp_g, &kbuf = ctx->pp_k;
  SBO_REQUIRE(gp >= 0 && gp < ctx->ms.G, "gp index out of range");
  SBO_TRY(points_common(ctx, m, x, tmp, xbuf));
  const ModelSpec& ms = ctx->ms;
  SBO_TRY(sbo_ensure(ctx, gbuf, sizeof(double) * (size_t)ms.d * m));
  const long long P = chunk_points(ctx, ms, m);
  SBO_TRY(sbo_ensure(ctx, kbuf, sizeof(double) * (size_t)ms.G * ms.npad * P));
  for (long long p0 = 0; p0 < m; p0 += P) {
    const int valid = (int)((m - p0) < P ? (m - p0) : P);
    SBO_TRY(crosscov_dispatch(ctx, tmp, p0, (int)P, valid, (double*)kbuf.p, nullptr, m, nullptr, (double*)gbuf.p, gp));
  }
  SBO_CUDA(cudaMemcpyAsync(grad, gbuf.p, sizeof(double) * (size_t)ms.d * m, cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}
