// batch.cu -- batch SafeOpt and GoOSE acquisition: q safe query points per step by hallucinated variance downdates of the
// objective GP (GP-BUCB-style; include/sbo_b200.h states the semantics).  All FP64, GP 0 only, normalised units:
//   k_batch_row     one CTA per pick: x_b from its global index, k_b = k(X, x_b), u_b = W^T (W k_b) = K^-1 k_b,
//                   row b of A = [c(x_i, x_j)] + sn I against the stored k / u of the earlier picks, row b of R (A = R R^T)
//   k_batch_update  grid over the candidates C = M u E: c(p, x_b) = k(p, x_b) - k(X, p) . u_b (X staged in shared memory in
//                   tiles, as the posterior kernels do), w_b(p) = (c - sum_{j<b} R_bj w_j(p)) / R_bb, v(p) -= w_b(p)^2 Ystd0^2
//                   (clamped at 0), and a fused arg-max (value, global index) over M and over E into block partials;
//                   b < 0: load v = var_0 and the membership bits instead
//   k_batch_choose  one CTA: reduce the partials, apply the pick rule (test/test_SafeOpt.py:153-158), write the record and
//                   the chosen global index to device memory, where the next k_batch_row reads it
// One GPU: 3 launches per pick and one copy to the host at the end.  v is kept in raw units (the step's var_0 as it is), so
// pick 1 reduces exactly the values the step reduced.
// GoOSE (C = S u T): k_batch_update<GOOSE> reduces lcb_0 = lcb_of(mean_0, v, beta) to a masked arg-min over S_b and T_b (the
// flag byte holds membership and "used" bits); k_goose_choose applies test/test_GoOSE.py:158-162, k_goose_nearest finds
// the point of S_b nearest to an explore pick's target, k_goose_finish writes the pick and retires its slot and the
// served target's slot.  One GPU: 5 launches per pick (the last pick needs 3), one copy to the host at the end.
#include "common.cuh"
#include <math.h>
#include <algorithm>

#define BT_THREADS 128
#define BT_JT 128
#define BT_ROW_THREADS 1024
#define BT_CHOOSE_THREADS 1024

struct BatchPart { double vm; long long im; double ve; long long ie; };
// GoOSE: bits of the per-candidate flag byte, and the decision of the current pick (device memory, after the records)
enum : uint8_t { GF_S = 1, GF_T = 2, GF_S_USED = 4, GF_T_USED = 8 };
struct GooseState { long long target; int explore, pad; long long near_idx; double near_d2; };
static_assert(sizeof(sbo_goose_batch_pick) >= sizeof(BatchRec), "the record area holds either kind of record");

// device pointers of the pick-side state (ctx->bt_pick): sel[q], rec[q] (BatchRec or sbo_goose_batch_pick), GooseState,
// R[q][q], xB[q][SBO_MAX_D], kB[q][npad], uB[q][npad], t[npad]
struct PickPtrs {
  long long* sel;
  BatchRec* rec;
  double *R, *xB, *kB, *uB, *t;
};
static size_t pick_bytes(int q, int npad) {
  return sizeof(long long) * q + sizeof(sbo_goose_batch_pick) * q + sizeof(GooseState) +
         sizeof(double) * ((size_t)q * q + (size_t)q * SBO_MAX_D + (2 * (size_t)q + 1) * npad);
}
static PickPtrs pick_ptrs(sbo_ctx* ctx) {
  const int q = ctx->bt.q, np = ctx->ms.npad;
  PickPtrs p;
  p.sel = (long long*)ctx->bt_pick.p;
  p.rec = (BatchRec*)(p.sel + q);
  p.R = (double*)((char*)p.rec + sizeof(sbo_goose_batch_pick) * q + sizeof(GooseState));
  p.xB = p.R + (size_t)q * q;
  p.kB = p.xB + (size_t)q * SBO_MAX_D;
  p.uB = p.kB + (size_t)q * np;
  p.t = p.uB + (size_t)q * np;
  return p;
}
static sbo_goose_batch_pick* goose_recs(const PickPtrs& p) { return (sbo_goose_batch_pick*)p.rec; }
static GooseState* goose_state(sbo_ctx* ctx, const PickPtrs& p) { return (GooseState*)(goose_recs(p) + ctx->bt.q); }

__device__ __forceinline__ double warp_sum(double s) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
  return s;
}

template <int D>
__device__ __forceinline__ double scaled_dist(const double* a, const double* b, const double* iell) {
  double s = 0.0;
#pragma unroll
  for (int k = 0; k < D; ++k) { const double df = a[k] - b[k]; s += df * df * iell[k]; }
  return s;
}

// C = M u (union of the expander masks)
__global__ void __launch_bounds__(256)
k_batch_union(long long nw, int n_exp, const uint32_t* __restrict__ m_min, const uint32_t* __restrict__ m_exp, uint32_t* __restrict__ out) {
  const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nw) return;
  uint32_t u = m_min[w];
  for (int c = 0; c < n_exp; ++c) u |= m_exp[(size_t)c * nw + w];
  out[w] = u;
}

template <int D, class KC>
__global__ void __launch_bounds__(BT_ROW_THREADS)
k_batch_row(ModelSpec ms, GridSpec gs, int b, int q, PickPtrs pp) {
  __shared__ double xn[SBO_MAX_D];
  __shared__ double a[SBO_BATCH_MAX_Q];
  const KC kc(ms.kernel);
  const int n = ms.n, np = ms.npad;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = BT_ROW_THREADS / 32;
  const double sf2 = ms.sf2[0];
  double iell[D];
#pragma unroll
  for (int k = 0; k < D; ++k) iell[k] = ms.inv_ell[0][k];
  if (tid == 0) {
    double x[SBO_MAX_D];
    point_coords(gs, pp.sel[b], x);
#pragma unroll
    for (int k = 0; k < D; ++k) {
      xn[k] = (x[k] - ms.Xmean[k]) / ms.Xstd[k];                     // GP_Safe.py:326
      pp.xB[(size_t)b * SBO_MAX_D + k] = xn[k];
    }
  }
  __syncthreads();
  double* kb = pp.kB + (size_t)b * np;
  double* ub = pp.uB + (size_t)b * np;
  for (int j = tid; j < n; j += BT_ROW_THREADS) kb[j] = kc.value(scaled_dist<D>(xn, ms.Xn + (size_t)j * D, iell), sf2);
  __syncthreads();
  // t = W k_b: one warp per row of the lower-triangular W
  for (int i = warp; i < n; i += NW) {
    const double* wr = ms.W + (size_t)i * np;
    double s = 0.0;
    for (int j = lane; j <= i; j += 32) s = fma(wr[j], kb[j], s);
    s = warp_sum(s);
    if (lane == 0) pp.t[i] = s;
  }
  __syncthreads();
  // u_b = W^T t: one thread per column; a warp reads rows from its first column on (W is zero above the diagonal), coalesced
  for (int j = tid; j < n; j += BT_ROW_THREADS) {
    double s = 0.0;
    for (int i = j - lane; i < n; ++i) s = fma(ms.W[(size_t)i * np + j], pp.t[i], s);
    ub[j] = s;
  }
  __syncthreads();
  // row b of A: c(x_b, x_j) = k(x_b, x_j) - k_b . u_j, plus sn on the diagonal; one warp per earlier pick
  for (int j = warp; j <= b; j += NW) {
    const double* uj = pp.uB + (size_t)j * np;
    double s = 0.0;
    for (int l = lane; l < n; l += 32) s = fma(kb[l], uj[l], s);
    s = warp_sum(s);
    if (lane == 0) a[j] = kc.value(scaled_dist<D>(xn, pp.xB + (size_t)j * SBO_MAX_D, iell), sf2) - s + (j == b ? ms.sn2[0] : 0.0);
  }
  __syncthreads();
  // row b of R by forward substitution; the Schur complement of A = C + sn I is >= sn (C is PSD): the floor only absorbs rounding
  if (warp == 0) {
    const double* R = pp.R;
    for (int j = 0; j < b; ++j) {
      double s = 0.0;
      for (int k = lane; k < j; k += 32) s = fma(a[k], R[(size_t)j * q + k], s);
      s = warp_sum(s);
      const double r = (a[j] - s) / R[(size_t)j * q + j];
      __syncwarp();
      if (lane == 0) a[j] = r;
      __syncwarp();
    }
    double s = 0.0;
    for (int k = lane; k < b; k += 32) s = fma(a[k], a[k], s);
    s = warp_sum(s);
    __syncwarp();
    if (lane == 0) a[b] = sqrt(fmax(a[b] - s, ms.sn2[0]));
    __syncwarp();
    for (int k = lane; k <= b; k += 32) pp.R[(size_t)b * q + k] = a[k];
  }
}

// SafeOpt: m_min / m_exp = M and the expander masks, arg-max of v over M and E.  GOOSE: the same arguments carry S and the
// target masks, and the reduction is the arg-min of lcb_0 over S_b and T_b (mean0 = the step's mean of GP 0, raw units).
template <int D, class KC, bool GOOSE>
__global__ void __launch_bounds__(BT_THREADS)
k_batch_update(ModelSpec ms, GridSpec gs, long long nc, int b, int q, const long long* __restrict__ cidx, uint8_t* __restrict__ flags,
               const uint32_t* __restrict__ m_min, const uint32_t* __restrict__ m_exp, int n_exp, long long nw,
               const double* __restrict__ var0, double* __restrict__ v, double* __restrict__ w, PickPtrs pp,
               BatchPart* __restrict__ part, const double* __restrict__ mean0, double beta) {
  __shared__ double Xs[BT_JT * D];
  __shared__ double Us[BT_JT];
  __shared__ double Rs[SBO_BATCH_MAX_Q];
  __shared__ ArgVal redm[BT_THREADS / 32], rede[BT_THREADS / 32];
  const KC kc(ms.kernel);
  const long long p = (long long)blockIdx.x * BT_THREADS + threadIdx.x;
  const bool ok = p < nc;
  const long long lp = ok ? cidx[p] : 0;
  const long long gp = shard_global(gs, lp);
  double vv = 0.0;
  uint8_t f = 0;
  if (b < 0) {                                  // initial state: the step's var_0 (raw units) and the membership bits
    if (ok) {
      vv = var0[lp];
      const uint32_t bit = 1u << (lp & 31);
      const long long wd = lp >> 5;
      f = (m_min[wd] & bit) ? 1 : 0;
      for (int c = 0; c < n_exp; ++c)
        if (m_exp[(size_t)c * nw + wd] & bit) f |= 2;
      flags[p] = f;
      v[p] = vv;
    }
  } else {
    const double sf2 = ms.sf2[0];
    double xn[D], iell[D];
#pragma unroll
    for (int k = 0; k < D; ++k) iell[k] = ms.inv_ell[0][k];
    if (ok) {
      double x[SBO_MAX_D];
      point_coords(gs, gp, x);
#pragma unroll
      for (int k = 0; k < D; ++k) xn[k] = (x[k] - ms.Xmean[k]) / ms.Xstd[k];
    } else {
#pragma unroll
      for (int k = 0; k < D; ++k) xn[k] = 0.0;
    }
    for (int j = threadIdx.x; j <= b; j += BT_THREADS) Rs[j] = pp.R[(size_t)b * q + j];
    const double* ub = pp.uB + (size_t)b * ms.npad;
    double acc = 0.0;                           // k(X, p) . u_b
    for (int j0 = 0; j0 < ms.n; j0 += BT_JT) {
      __syncthreads();
      for (int e = threadIdx.x; e < BT_JT * D; e += BT_THREADS) Xs[e] = (j0 * D + e < ms.n * D) ? ms.Xn[(size_t)j0 * D + e] : 0.0;
      for (int e = threadIdx.x; e < BT_JT; e += BT_THREADS) Us[e] = (j0 + e < ms.n) ? ub[j0 + e] : 0.0;
      __syncthreads();
      const int jn = min(BT_JT, ms.n - j0);
      if (ok)
        for (int j = 0; j < jn; ++j) acc = fma(kc.value(scaled_dist<D>(xn, Xs + j * D, iell), sf2), Us[j], acc);
    }
    if (ok) {
      const double c = kc.value(scaled_dist<D>(xn, pp.xB + (size_t)b * SBO_MAX_D, iell), sf2) - acc;
      double corr = 0.0;
      for (int j = 0; j < b; ++j) corr = fma(Rs[j], w[(size_t)j * nc + p], corr);
      const double wb = (c - corr) / Rs[b];
      w[(size_t)b * nc + p] = wb;
      vv = fmax(0.0, v[p] - wb * wb * (ms.Ystd[0] * ms.Ystd[0]));
      v[p] = vv;
      f = flags[p];
    }
  }
  if constexpr (GOOSE) {
    const ArgVal none = {INFINITY, SBO_IDX_NONE};
    const double l = ok ? lcb_of(mean0[lp], vv, beta) : 0.0;             // b < 0: exactly the step's lcb_0
    ArgVal as = ((f & (GF_S | GF_S_USED)) == GF_S) ? ArgVal{l, gp} : none;
    ArgVal at = ((f & (GF_T | GF_T_USED)) == GF_T) ? ArgVal{l, gp} : none;
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) {
      as = argmin2(as, shfl_xor_argval(as, m));
      at = argmin2(at, shfl_xor_argval(at, m));
    }
    if ((threadIdx.x & 31) == 0) { redm[threadIdx.x >> 5] = as; rede[threadIdx.x >> 5] = at; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int k = 1; k < BT_THREADS / 32; ++k) { as = argmin2(as, redm[k]); at = argmin2(at, rede[k]); }
      part[blockIdx.x] = BatchPart{as.v, as.i, at.v, at.i};
    }
  } else {
    const ArgVal none = {-INFINITY, SBO_IDX_NONE};
    ArgVal am = (f & 1) ? ArgVal{vv, gp} : none;
    ArgVal ae = (f & 2) ? ArgVal{vv, gp} : none;
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) {
      am = argmax2(am, shfl_xor_argval(am, m));
      ae = argmax2(ae, shfl_xor_argval(ae, m));
    }
    if ((threadIdx.x & 31) == 0) { redm[threadIdx.x >> 5] = am; rede[threadIdx.x >> 5] = ae; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int k = 1; k < BT_THREADS / 32; ++k) { am = argmax2(am, redm[k]); ae = argmax2(ae, rede[k]); }
      part[blockIdx.x] = BatchPart{am.v, am.i, ae.v, ae.i};
    }
  }
}

__global__ void __launch_bounds__(BT_CHOOSE_THREADS)
k_batch_choose(const BatchPart* __restrict__ part, int nparts, int b, long long* __restrict__ sel, BatchRec* __restrict__ rec) {
  __shared__ ArgVal redm[BT_CHOOSE_THREADS / 32], rede[BT_CHOOSE_THREADS / 32];
  const ArgVal none = {-INFINITY, SBO_IDX_NONE};
  ArgVal am = none, ae = none;
  for (int i = threadIdx.x; i < nparts; i += BT_CHOOSE_THREADS) {
    const BatchPart pt = part[i];
    am = argmax2(am, ArgVal{pt.vm, pt.im});
    ae = argmax2(ae, ArgVal{pt.ve, pt.ie});
  }
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) {
    am = argmax2(am, shfl_xor_argval(am, m));
    ae = argmax2(ae, shfl_xor_argval(ae, m));
  }
  if ((threadIdx.x & 31) == 0) { redm[threadIdx.x >> 5] = am; rede[threadIdx.x >> 5] = ae; }
  __syncthreads();
  if (threadIdx.x != 0) return;
  for (int k = 1; k < BT_CHOOSE_THREADS / 32; ++k) { am = argmax2(am, redm[k]); ae = argmax2(ae, rede[k]); }
  const bool hm = am.i != SBO_IDX_NONE, he = ae.i != SBO_IDX_NONE;
  BatchRec r;
  r.vmin = hm ? am.v : 0.0; r.imin = hm ? am.i : -1;
  r.vexp = he ? ae.v : 0.0; r.iexp = he ? ae.i : -1;
  const bool take_min = hm && (!he || sqrt(am.v) > sqrt(ae.v));         // test/test_SafeOpt.py:153-158, empty set yields
  r.idx = take_min ? r.imin : r.iexp;
  r.from_exp = (!take_min && he) ? 1 : 0;
  r.pad = 0;
  rec[b] = r;
  sel[b] = r.idx;
}

// GoOSE pick b: reduce the partials of k_batch_update<GOOSE> and apply test/test_GoOSE.py:158-162.  A safe pick is final here;
// an explore pick leaves its idx to k_goose_finish, after k_goose_nearest.  S_b empty: no pick (idx = -1).
__global__ void __launch_bounds__(BT_CHOOSE_THREADS)
k_goose_choose(const BatchPart* __restrict__ part, int nparts, int b, sbo_goose_batch_pick* __restrict__ rec, GooseState* __restrict__ gst) {
  __shared__ ArgVal reds[BT_CHOOSE_THREADS / 32], redt[BT_CHOOSE_THREADS / 32];
  const ArgVal none = {INFINITY, SBO_IDX_NONE};
  ArgVal as = none, at = none;
  for (int i = threadIdx.x; i < nparts; i += BT_CHOOSE_THREADS) {
    const BatchPart pt = part[i];
    as = argmin2(as, ArgVal{pt.vm, pt.im});
    at = argmin2(at, ArgVal{pt.ve, pt.ie});
  }
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) {
    as = argmin2(as, shfl_xor_argval(as, m));
    at = argmin2(at, shfl_xor_argval(at, m));
  }
  if ((threadIdx.x & 31) == 0) { reds[threadIdx.x >> 5] = as; redt[threadIdx.x >> 5] = at; }
  __syncthreads();
  if (threadIdx.x != 0) return;
  for (int k = 1; k < BT_CHOOSE_THREADS / 32; ++k) { as = argmin2(as, reds[k]); at = argmin2(at, redt[k]); }
  const bool hs = as.i != SBO_IDX_NONE, ht = at.i != SBO_IDX_NONE;
  sbo_goose_batch_pick r;
  r.safe_lcb = hs ? as.v : INFINITY; r.safe_idx = hs ? as.i : -1;
  r.target_lcb = ht ? at.v : INFINITY; r.target_idx = ht ? at.i : -1;
  const bool explore = hs && ht && !(as.v <= at.v);
  r.idx = explore ? -1 : r.safe_idx;
  r.explore = explore ? 1 : 0;
  r.pad = 0;
  r.dist = 0.0;
  rec[b] = r;
  gst->target = explore ? r.target_idx : -1;
  gst->explore = r.explore;
}

// explore pick: (squared distance, global index) to the target over S_b into block partials, the expression of
// k_argreduce<SBO_ARGMIN_DIST> (sets.cu); returns at once for a safe pick
__global__ void __launch_bounds__(BT_THREADS)
k_goose_nearest(GridSpec gs, long long nc, const long long* __restrict__ cidx, const uint8_t* __restrict__ flags,
                const GooseState* __restrict__ gst, BatchPart* __restrict__ part) {
  __shared__ ArgVal red[BT_THREADS / 32];
  if (!gst->explore) return;
  const long long p = (long long)blockIdx.x * BT_THREADS + threadIdx.x;
  ArgVal a = {INFINITY, SBO_IDX_NONE};
  if (p < nc && (flags[p] & (GF_S | GF_S_USED)) == GF_S) {
    const long long gp = shard_global(gs, cidx[p]);
    double x[SBO_MAX_D], t[SBO_MAX_D];
    point_coords(gs, gp, x);
    point_coords(gs, gst->target, t);
    double v = 0.0;
    for (int k = 0; k < gs.d; ++k) { const double df = x[k] - t[k]; v = __dadd_rn(v, __dmul_rn(df, df)); }
    a = ArgVal{v, gp};
  }
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) a = argmin2(a, shfl_xor_argval(a, m));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < BT_THREADS / 32; ++k) a = argmin2(a, red[k]);
    part[blockIdx.x] = BatchPart{a.v, a.i, 0.0, SBO_IDX_NONE};
  }
}

// slot of GLOBAL index g among the compacted candidates (ascending local index, so ascending global index), -1 if absent
__device__ long long candidate_slot(const GridSpec& gs, const long long* cidx, long long nc, long long g) {
  long long lo = 0, hi = nc;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (shard_global(gs, cidx[mid]) < g) lo = mid + 1; else hi = mid;
  }
  return (lo < nc && shard_global(gs, cidx[lo]) == g) ? lo : -1;
}

enum { GOOSE_FINISH_PICK = 0, GOOSE_FINISH_NEAREST = 1, GOOSE_FINISH_COMMIT = 2 };
// PICK (one GPU): an explore pick takes the nearest point of S_b; then sel[b] = the pick and both slots are retired.
// NEAREST (staged): only the local nearest point, into gst->near_idx / near_d2.  COMMIT (staged): retire sel[b] and the
// served target gst->target (set by the host).
__global__ void __launch_bounds__(BT_CHOOSE_THREADS)
k_goose_finish(const BatchPart* __restrict__ near, int nparts, int b, int mode, GridSpec gs, long long nc,
               const long long* __restrict__ cidx, uint8_t* __restrict__ flags, long long* __restrict__ sel,
               sbo_goose_batch_pick* __restrict__ rec, GooseState* __restrict__ gst) {
  __shared__ ArgVal red[BT_CHOOSE_THREADS / 32];
  if (mode != GOOSE_FINISH_COMMIT && gst->explore) {
    ArgVal a = {INFINITY, SBO_IDX_NONE};
    for (int i = threadIdx.x; i < nparts; i += BT_CHOOSE_THREADS) a = argmin2(a, ArgVal{near[i].vm, near[i].im});
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) a = argmin2(a, shfl_xor_argval(a, m));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int k = 1; k < BT_CHOOSE_THREADS / 32; ++k) a = argmin2(a, red[k]);
      const bool h = a.i != SBO_IDX_NONE;
      gst->near_idx = h ? a.i : -1;
      gst->near_d2 = h ? a.v : INFINITY;
      if (mode == GOOSE_FINISH_PICK) { rec[b].idx = gst->near_idx; rec[b].dist = sqrt(gst->near_d2); }
    }
  }
  if (mode == GOOSE_FINISH_NEAREST || threadIdx.x != 0) return;
  if (mode == GOOSE_FINISH_PICK) sel[b] = rec[b].idx;
  const long long s = candidate_slot(gs, cidx, nc, sel[b]);
  if (s >= 0) flags[s] |= GF_S_USED;
  if (gst->explore) {
    const long long t = candidate_slot(gs, cidx, nc, gst->target);
    if (t >= 0) flags[t] |= GF_T_USED;
  }
}

// ---------------------------------------------------------------------------------------------
// host drivers
// ---------------------------------------------------------------------------------------------
static int batch_valid(sbo_ctx* ctx) {
  SBO_REQUIRE(ctx->bt.prepared && !ctx->bt.goose && ctx->have_exp,
              "no prepared batch for the current SafeOpt pair stage (call sbo_batch_prepare after the step)");
  return SBO_OK;
}
static int goose_valid(sbo_ctx* ctx) {
  SBO_REQUIRE(ctx->bt.prepared && ctx->bt.goose && ctx->have_tgt,
              "no prepared GoOSE batch for the current GoOSE target stage (call sbo_goose_batch_prepare after the step)");
  return SBO_OK;
}

static int launch_row(sbo_ctx* ctx, int b) {
  const PickPtrs pp = pick_ptrs(ctx);
  with_int<1, SBO_MAX_D>(ctx->ms.d, [&](auto D) { with_kernel(ctx->ms.kernel, [&](auto kc) {
    k_batch_row<D, decltype(kc)><<<1, BT_ROW_THREADS, 0, ctx->stream>>>(ctx->ms, ctx->gs, b, ctx->bt.q, pp);
  }); });
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

// b < 0: initial state; else the downdate by pick b and the partials for pick b + 1
static int launch_update(sbo_ctx* ctx, int b) {
  const BatchStage& bs = ctx->bt;
  if (bs.nc == 0) return SBO_OK;
  const PickPtrs pp = pick_ptrs(ctx);
  const int n_exp = ctx->ms.G > 1 ? ctx->ms.G - 1 : 1;
  // GoOSE: S and the target masks take the places of M and the expander masks
  const uint32_t* m_a = (const uint32_t*)(bs.goose ? ctx->m_safe.p : ctx->m_min.p);
  const uint32_t* m_b = (const uint32_t*)(bs.goose ? ctx->m_tgt.p : ctx->m_exp.p);
  with_int<1, SBO_MAX_D>(ctx->ms.d, [&](auto D) { with_kernel(ctx->ms.kernel, [&](auto kc) { with_flag(bs.goose, [&](auto GOOSE) {
    k_batch_update<D, decltype(kc), GOOSE><<<bs.nparts, BT_THREADS, 0, ctx->stream>>>(
        ctx->ms, ctx->gs, bs.nc, b, bs.q, (const long long*)ctx->bt_idx.p, (uint8_t*)ctx->bt_flag.p, m_a, m_b, n_exp, mask_words(ctx),
        (const double*)ctx->var.p, (double*)ctx->bt_v.p, (double*)ctx->bt_w.p, pp, (BatchPart*)ctx->bt_part.p,
        (const double*)ctx->mean.p, ctx->beta);
  }); }); });
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

static int launch_choose(sbo_ctx* ctx, int b) {
  const PickPtrs pp = pick_ptrs(ctx);
  k_batch_choose<<<1, BT_CHOOSE_THREADS, 0, ctx->stream>>>((const BatchPart*)ctx->bt_part.p, (int)(ctx->bt.nc > 0 ? ctx->bt.nparts : 0), b,
                                                           pp.sel, pp.rec);
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

// the candidates C = a u (union of the n_exp masks b), compacted, and the initial state (v = var_0, membership bits)
static int prepare_candidates(sbo_ctx* ctx, int q, bool goose, long long* n_candidates) {
  BatchStage& bs = ctx->bt;
  stage_changed(ctx, Change::BATCH);
  bs.goose = goose; bs.b = 0;
  const long long count = ctx->gs.count, nw = mask_words(ctx);
  const int n_exp = ctx->ms.G > 1 ? ctx->ms.G - 1 : 1;
  SBO_TRY(sbo_ensure(ctx, ctx->bt_mask, sizeof(uint32_t) * (size_t)nw));
  k_batch_union<<<(unsigned)cdiv(nw, 256), 256, 0, ctx->stream>>>(nw, n_exp, (const uint32_t*)(goose ? ctx->m_safe.p : ctx->m_min.p),
                                                                  (const uint32_t*)(goose ? ctx->m_tgt.p : ctx->m_exp.p),
                                                                  (uint32_t*)ctx->bt_mask.p);
  SBO_LAUNCH_CHECK();
  long long nc = 0;
  SBO_TRY(compact_mask(ctx, (const uint32_t*)ctx->bt_mask.p, count, ctx->bt_idx, &nc));
  bs.q = q; bs.nc = nc;
  bs.nparts = (int)cdiv(nc > 0 ? nc : 1, BT_THREADS);
  SBO_TRY(sbo_ensure(ctx, ctx->bt_flag, (size_t)(nc > 0 ? nc : 1)));
  SBO_TRY(sbo_ensure(ctx, ctx->bt_v, sizeof(double) * (size_t)(nc > 0 ? nc : 1)));
  SBO_TRY(sbo_ensure(ctx, ctx->bt_w, sizeof(double) * (size_t)q * (nc > 0 ? nc : 1)));
  // GoOSE: a second set of partials for k_goose_nearest, so that the staged calls may interleave
  SBO_TRY(sbo_ensure(ctx, ctx->bt_part, sizeof(BatchPart) * (size_t)bs.nparts * (goose ? 2 : 1)));
  SBO_TRY(sbo_ensure(ctx, ctx->bt_pick, pick_bytes(q, ctx->ms.npad)));
  SBO_TRY(launch_update(ctx, -1));
  stage_changed(ctx, Change::BATCH_PREPARED);
  if (n_candidates) *n_candidates = nc;
  return SBO_OK;
}

int batch_prepare(sbo_ctx* ctx, int q, long long* n_candidates) {
  SBO_REQUIRE(q >= 1 && q <= SBO_BATCH_MAX_Q, "batch size q out of range (1..256)");
  SBO_REQUIRE(ctx->have_post && ctx->have_sets2 && ctx->have_exp,
              "batch acquisition needs a SafeOpt pair stage (sbo_expander after sbo_sets, or a sharded SafeOpt step) since the last "
              "model, grid, shard, posterior or set change; a GoOSE target stage does not provide one");
  return prepare_candidates(ctx, q, false, n_candidates);
}

int batch_local(sbo_ctx* ctx, BatchRec* out) {
  SBO_TRY(batch_valid(ctx));
  SBO_REQUIRE(out != nullptr, "null result");
  SBO_REQUIRE(ctx->bt.b < ctx->bt.q, "all q picks of the batch are committed");
  const int b = ctx->bt.b;
  SBO_TRY(launch_choose(ctx, b));
  SBO_CUDA(cudaMemcpyAsync(out, pick_ptrs(ctx).rec + b, sizeof(BatchRec), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}

int batch_commit(sbo_ctx* ctx, long long global_idx) {
  SBO_TRY(batch_valid(ctx));
  SBO_REQUIRE(ctx->bt.b < ctx->bt.q, "all q picks of the batch are committed");
  SBO_REQUIRE(global_idx >= 0 && global_idx < ctx->gs.N, "global index out of range");
  const int b = ctx->bt.b;
  SBO_CUDA(cudaMemcpyAsync(pick_ptrs(ctx).sel + b, &global_idx, sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
  SBO_TRY(launch_row(ctx, b));
  SBO_TRY(launch_update(ctx, b));
  ctx->bt.b = b + 1;
  return SBO_OK;
}

void batch_pick_of(const BatchRec& r, sbo_batch_pick* out) {
  out->idx = r.idx;
  out->from_expander = r.from_exp;
  out->pad = 0;
  out->std_min = r.imin >= 0 ? sqrt(r.vmin) : 0.0;
  out->idx_min = r.imin;
  out->std_exp = r.iexp >= 0 ? sqrt(r.vexp) : 0.0;
  out->idx_exp = r.iexp;
}

// ---- GoOSE -------------------------------------------------------------------------------------
static int launch_goose_choose(sbo_ctx* ctx, int b) {
  const PickPtrs pp = pick_ptrs(ctx);
  k_goose_choose<<<1, BT_CHOOSE_THREADS, 0, ctx->stream>>>((const BatchPart*)ctx->bt_part.p, (int)(ctx->bt.nc > 0 ? ctx->bt.nparts : 0), b,
                                                           goose_recs(pp), goose_state(ctx, pp));
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

static int launch_goose_nearest(sbo_ctx* ctx) {
  const BatchStage& bs = ctx->bt;
  if (bs.nc == 0) return SBO_OK;
  const PickPtrs pp = pick_ptrs(ctx);
  k_goose_nearest<<<bs.nparts, BT_THREADS, 0, ctx->stream>>>(ctx->gs, bs.nc, (const long long*)ctx->bt_idx.p, (const uint8_t*)ctx->bt_flag.p,
                                                             goose_state(ctx, pp), (BatchPart*)ctx->bt_part.p + bs.nparts);
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

static int launch_goose_finish(sbo_ctx* ctx, int b, int mode) {
  const BatchStage& bs = ctx->bt;
  const PickPtrs pp = pick_ptrs(ctx);
  k_goose_finish<<<1, BT_CHOOSE_THREADS, 0, ctx->stream>>>((const BatchPart*)ctx->bt_part.p + bs.nparts, (int)(bs.nc > 0 ? bs.nparts : 0), b, mode,
                                                           ctx->gs, bs.nc, (const long long*)ctx->bt_idx.p, (uint8_t*)ctx->bt_flag.p,
                                                           pp.sel, goose_recs(pp), goose_state(ctx, pp));
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

int goose_batch_prepare(sbo_ctx* ctx, int q, long long* n_candidates) {
  SBO_REQUIRE(q >= 1 && q <= SBO_BATCH_MAX_Q, "batch size q out of range (1..256)");
  SBO_REQUIRE(ctx->have_post && ctx->have_sets && ctx->have_tgt,
              "GoOSE batch acquisition needs a GoOSE target stage (sbo_goose_target after sbo_sets_pass1, or a sharded GoOSE step) "
              "since the last model, grid, shard, posterior or set change; a SafeOpt pair stage does not provide one");
  return prepare_candidates(ctx, q, true, n_candidates);
}

int goose_batch_local(sbo_ctx* ctx, sbo_goose_batch_pick* out) {
  SBO_TRY(goose_valid(ctx));
  SBO_REQUIRE(out != nullptr, "null result");
  SBO_REQUIRE(ctx->bt.b < ctx->bt.q, "all q picks of the batch are committed");
  const int b = ctx->bt.b;
  SBO_TRY(launch_goose_choose(ctx, b));
  SBO_CUDA(cudaMemcpyAsync(out, goose_recs(pick_ptrs(ctx)) + b, sizeof(*out), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}

int goose_batch_nearest(sbo_ctx* ctx, long long target, long long* idx, double* dist2) {
  SBO_TRY(goose_valid(ctx));
  SBO_REQUIRE(idx && dist2, "null result");
  SBO_REQUIRE(ctx->bt.b < ctx->bt.q, "all q picks of the batch are committed");
  SBO_REQUIRE(target >= 0 && target < ctx->gs.N, "global index out of range");
  const PickPtrs pp = pick_ptrs(ctx);
  GooseState st{target, 1, 0, -1, INFINITY};
  SBO_CUDA(cudaMemcpyAsync(goose_state(ctx, pp), &st, sizeof(st), cudaMemcpyHostToDevice, ctx->stream));
  SBO_TRY(launch_goose_nearest(ctx));
  SBO_TRY(launch_goose_finish(ctx, ctx->bt.b, GOOSE_FINISH_NEAREST));
  SBO_CUDA(cudaMemcpyAsync(&st, goose_state(ctx, pp), sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  *idx = st.near_idx;
  *dist2 = st.near_d2;
  return SBO_OK;
}

int goose_batch_commit(sbo_ctx* ctx, long long pick, long long served_target) {
  SBO_TRY(goose_valid(ctx));
  SBO_REQUIRE(ctx->bt.b < ctx->bt.q, "all q picks of the batch are committed");
  SBO_REQUIRE(pick >= 0 && pick < ctx->gs.N, "global index out of range");
  SBO_REQUIRE(served_target >= -1 && served_target < ctx->gs.N, "served target index out of range");
  const int b = ctx->bt.b;
  const PickPtrs pp = pick_ptrs(ctx);
  const GooseState st{served_target, served_target >= 0 ? 1 : 0, 0, -1, INFINITY};
  SBO_CUDA(cudaMemcpyAsync(pp.sel + b, &pick, sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
  SBO_CUDA(cudaMemcpyAsync(goose_state(ctx, pp), &st, sizeof(st), cudaMemcpyHostToDevice, ctx->stream));
  SBO_TRY(launch_goose_finish(ctx, b, GOOSE_FINISH_COMMIT));
  SBO_TRY(launch_row(ctx, b));
  SBO_TRY(launch_update(ctx, b));
  ctx->bt.b = b + 1;
  return SBO_OK;
}

extern "C" {

int sbo_safeopt_batch(sbo_ctx* ctx, int q, sbo_batch_pick* picks, int* n_picked) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  SBO_REQUIRE(picks && n_picked, "null result");
  long long nc = 0;
  SBO_TRY(batch_prepare(ctx, q, &nc));
  stage_changed(ctx, Change::BATCH);            // the whole batch runs here; the staged calls need their own prepare
  std::vector<BatchRec> rec(q);
  if (nc == 0) {                                // M and E are both empty, and stay so
    SBO_TRY(launch_choose(ctx, 0));
    SBO_CUDA(cudaMemcpyAsync(rec.data(), pick_ptrs(ctx).rec, sizeof(BatchRec), cudaMemcpyDeviceToHost, ctx->stream));
    SBO_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < q; ++b) batch_pick_of(rec[0], &picks[b]);
    *n_picked = 0;
    return SBO_OK;
  }
  for (int b = 0; b < q; ++b) {                 // no host synchronisation: k_batch_row reads the pick from device memory
    SBO_TRY(launch_choose(ctx, b));
    if (b + 1 < q) {
      SBO_TRY(launch_row(ctx, b));
      SBO_TRY(launch_update(ctx, b));
    }
  }
  SBO_CUDA(cudaMemcpyAsync(rec.data(), pick_ptrs(ctx).rec, sizeof(BatchRec) * q, cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int b = 0; b < q; ++b) batch_pick_of(rec[b], &picks[b]);
  *n_picked = q;                                // C is not empty: every pick has a candidate
  return SBO_OK;
}

int sbo_batch_prepare(sbo_ctx* ctx, int q, int64_t* n_candidates_local) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  long long nc = 0;
  SBO_TRY(batch_prepare(ctx, q, &nc));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  if (n_candidates_local) *n_candidates_local = nc;
  return SBO_OK;
}

int sbo_batch_local(sbo_ctx* ctx, sbo_batch_pick* local_optima) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  SBO_REQUIRE(local_optima != nullptr, "null result");
  BatchRec r;
  SBO_TRY(batch_local(ctx, &r));
  batch_pick_of(r, local_optima);
  return SBO_OK;
}

int sbo_batch_commit(sbo_ctx* ctx, int64_t global_idx) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  SBO_TRY(batch_commit(ctx, global_idx));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}

int sbo_goose_batch(sbo_ctx* ctx, int q, sbo_goose_batch_pick* picks, int* n_picked) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  SBO_REQUIRE(picks && n_picked, "null result");
  SBO_TRY(goose_batch_prepare(ctx, q, nullptr));
  stage_changed(ctx, Change::BATCH);            // the whole batch runs here; the staged calls need their own prepare
  // every pick retires one point of S, and a pick exists while S_b is not empty: exactly min(q, |S|) picks
  const int n = (int)std::min<long long>(q, ctx->n_safe_local);
  sbo_goose_batch_pick* rec = goose_recs(pick_ptrs(ctx));
  if (n == 0) {                                 // S is empty: report the optima (T may not be empty), no pick
    SBO_TRY(launch_goose_choose(ctx, 0));
    SBO_CUDA(cudaMemcpyAsync(picks, rec, sizeof(*picks), cudaMemcpyDeviceToHost, ctx->stream));
    SBO_CUDA(cudaStreamSynchronize(ctx->stream));
    *n_picked = 0;
    return SBO_OK;
  }
  for (int b = 0; b < n; ++b) {                 // no host synchronisation: the kernels pass the pick on in device memory
    SBO_TRY(launch_goose_choose(ctx, b));
    SBO_TRY(launch_goose_nearest(ctx));
    SBO_TRY(launch_goose_finish(ctx, b, GOOSE_FINISH_PICK));
    if (b + 1 < n) {
      SBO_TRY(launch_row(ctx, b));
      SBO_TRY(launch_update(ctx, b));
    }
  }
  SBO_CUDA(cudaMemcpyAsync(picks, rec, sizeof(*picks) * n, cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  *n_picked = n;
  return SBO_OK;
}

int sbo_goose_batch_prepare(sbo_ctx* ctx, int q, int64_t* n_candidates_local) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  long long nc = 0;
  SBO_TRY(goose_batch_prepare(ctx, q, &nc));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  if (n_candidates_local) *n_candidates_local = nc;
  return SBO_OK;
}

int sbo_goose_batch_local(sbo_ctx* ctx, sbo_goose_batch_pick* local_optima) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  return goose_batch_local(ctx, local_optima);
}

int sbo_goose_batch_nearest(sbo_ctx* ctx, int64_t target_global_idx, int64_t* idx, double* dist2) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  long long li = -1;
  SBO_TRY(goose_batch_nearest(ctx, target_global_idx, &li, dist2));
  if (idx) *idx = li;
  return SBO_OK;
}

int sbo_goose_batch_commit(sbo_ctx* ctx, int64_t pick_global_idx, int64_t served_target_global_idx) {
  if (!ctx) return sbo_fail(nullptr, SBO_ERR_INVALID, "null context");
  cudaSetDevice(ctx->device);
  SBO_TRY(goose_batch_commit(ctx, pick_global_idx, served_target_global_idx));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  return SBO_OK;
}

}  // extern "C"
