// sets.cu -- confidence bounds, packed safe / unsafe / minimiser bitmasks and deterministic
// arg-reductions (warp-shuffle, lowest-index tie-break) over the local shard.
//   lcb/ucb              models/SafeOpt.py:34-45
//   S = {lcb_i >= 0}     SafeOpt.py:58-59, GoOSE.py:22-25   (strict '>' = plot mask, test_SafeOpt.py:337-338)
//   Z                    SafeOpt.py:73-77,109 (lcb_constraint_min returns the max; "<= 0")
//   min_S ucb_0          SafeOpt.py:47-51 ; min_S lcb_0  GoOSE.py:63-67
//   M, argmax var_0      SafeOpt.py:53-66
#include "common.cuh"
#include <math.h>

#define ST 256

struct SetsPartial {   // one per block
  double min_ucb; long long min_ucb_i;
  double min_lcb; long long min_lcb_i;
  long long n_safe, n_unsafe;
};
struct Pass2Partial {
  double max_var; long long max_var_i;
  long long n_min;
};
struct SetsDeviceResult {
  double min_ucb; long long min_ucb_i;
  double min_lcb; long long min_lcb_i;
  long long n_safe, n_unsafe;
  double max_var; long long max_var_i;
  long long n_min;
};

__device__ __forceinline__ ArgVal block_argmin(ArgVal a, ArgVal* sm) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) a = argmin2(a, shfl_xor_argval(a, m));
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x < 32) {
    ArgVal b = (threadIdx.x < (blockDim.x >> 5)) ? sm[threadIdx.x] : ArgVal{INFINITY, SBO_IDX_NONE};
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) b = argmin2(b, shfl_xor_argval(b, m));
    a = b;
  }
  __syncthreads();
  return a;   // valid in warp 0
}
__device__ __forceinline__ ArgVal block_argmax(ArgVal a, ArgVal* sm) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) a = argmax2(a, shfl_xor_argval(a, m));
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x < 32) {
    ArgVal b = (threadIdx.x < (blockDim.x >> 5)) ? sm[threadIdx.x] : ArgVal{-INFINITY, SBO_IDX_NONE};
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) b = argmax2(b, shfl_xor_argval(b, m));
    a = b;
  }
  __syncthreads();
  return a;
}
__device__ __forceinline__ long long block_sum_ll(long long v, long long* sm) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    long long b = (threadIdx.x < (blockDim.x >> 5)) ? sm[threadIdx.x] : 0;
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) b += __shfl_xor_sync(0xffffffffu, b, m);
    v = b;
  }
  __syncthreads();
  return v;
}

// pass 1: one thread per point, one ballot word per warp
__global__ void __launch_bounds__(ST)
k_sets_pass1(int G, long long count, GridSpec gs, const double* __restrict__ mean, const double* __restrict__ var,
             double beta, int rule, int strict, uint32_t* __restrict__ safe_w, uint32_t* __restrict__ unsafe_w,
             SetsPartial* __restrict__ part) {
  __shared__ ArgVal sm_av[ST / 32];
  __shared__ long long sm_ll[ST / 32];
  const long long p = (long long)blockIdx.x * ST + threadIdx.x;
  bool safe = false, unsafe = false;
  ArgVal u{INFINITY, SBO_IDX_NONE}, l{INFINITY, SBO_IDX_NONE};
  if (p < count) {
    safe = true;
    bool all_le = true, any_lt = false;
    for (int i = 1; i < G; ++i) {
      const double lcb = lcb_of(mean[(size_t)i * count + p], var[(size_t)i * count + p], beta);   // SafeOpt.py:40-45
      safe = safe && (strict ? (lcb > 0.0) : (lcb >= 0.0));
      all_le = all_le && (lcb <= 0.0);
      any_lt = any_lt || (lcb < 0.0);
    }
    unsafe = (G > 1) && (rule == SBO_UNSAFE_ALL ? all_le : any_lt);
    if (safe) {
      u = ArgVal{ucb_of(mean[p], var[p], beta), shard_global(gs, p)};
      l = ArgVal{lcb_of(mean[p], var[p], beta), shard_global(gs, p)};
    }
  }
  const uint32_t ws = __ballot_sync(0xffffffffu, safe), wu = __ballot_sync(0xffffffffu, unsafe);
  if ((threadIdx.x & 31) == 0 && p < count) { safe_w[p >> 5] = ws; unsafe_w[p >> 5] = wu; }
  u = block_argmin(u, sm_av);
  l = block_argmin(l, sm_av);
  const long long ns = block_sum_ll(safe ? 1 : 0, sm_ll);
  const long long nu = block_sum_ll(unsafe ? 1 : 0, sm_ll);
  if (threadIdx.x == 0) part[blockIdx.x] = SetsPartial{u.v, u.i, l.v, l.i, ns, nu};
}

__global__ void __launch_bounds__(ST) k_sets_final1(const SetsPartial* __restrict__ part, int nblocks, SetsDeviceResult* __restrict__ res) {
  __shared__ ArgVal sm_av[ST / 32];
  __shared__ long long sm_ll[ST / 32];
  ArgVal u{INFINITY, SBO_IDX_NONE}, l{INFINITY, SBO_IDX_NONE};
  long long ns = 0, nu = 0;
  for (int b = threadIdx.x; b < nblocks; b += ST) {
    u = argmin2(u, ArgVal{part[b].min_ucb, part[b].min_ucb_i});
    l = argmin2(l, ArgVal{part[b].min_lcb, part[b].min_lcb_i});
    ns += part[b].n_safe; nu += part[b].n_unsafe;
  }
  u = block_argmin(u, sm_av);
  l = block_argmin(l, sm_av);
  ns = block_sum_ll(ns, sm_ll);
  nu = block_sum_ll(nu, sm_ll);
  if (threadIdx.x == 0) {
    res->min_ucb = u.v; res->min_ucb_i = (u.i == SBO_IDX_NONE) ? -1 : u.i;
    res->min_lcb = l.v; res->min_lcb_i = (l.i == SBO_IDX_NONE) ? -1 : l.i;
    res->n_safe = ns; res->n_unsafe = nu;
  }
}

// pass 2: M = S and lcb_0 <= min_ucb0 ; argmax var_0 over M
__global__ void __launch_bounds__(ST)
k_sets_pass2(long long count, GridSpec gs, const double* __restrict__ mean, const double* __restrict__ var,
             double beta, double min_ucb0, const uint32_t* __restrict__ safe_w, uint32_t* __restrict__ min_w,
             Pass2Partial* __restrict__ part) {
  __shared__ ArgVal sm_av[ST / 32];
  __shared__ long long sm_ll[ST / 32];
  const long long p = (long long)blockIdx.x * ST + threadIdx.x;
  bool inM = false;
  ArgVal a{-INFINITY, SBO_IDX_NONE};
  if (p < count) {
    const bool safe = (safe_w[p >> 5] >> (p & 31)) & 1u;
    if (safe) {
      const double lcb0 = lcb_of(mean[p], var[p], beta);
      inM = lcb0 <= min_ucb0;                                    // SafeOpt.py:62
      if (inM) a = ArgVal{var[p], shard_global(gs, p)};                    // SafeOpt.py:55,65
    }
  }
  const uint32_t wm = __ballot_sync(0xffffffffu, inM);
  if ((threadIdx.x & 31) == 0 && p < count) min_w[p >> 5] = wm;
  a = block_argmax(a, sm_av);
  const long long nm = block_sum_ll(inM ? 1 : 0, sm_ll);
  if (threadIdx.x == 0) part[blockIdx.x] = Pass2Partial{a.v, a.i, nm};
}


// ---------------------------------------------------------------------------------------------
// Vectorised K2 (count % 4 == 0): persistent grid-stride CTAs, 4 consecutive points per thread read with 128-bit
// loads (2 x double2 per GP array), every load of a tile issued before the first use; one nibble of mask bits per
// thread, assembled into words by three xor-shuffles inside groups of 8 lanes.  HBM-bound: 16*G bytes per point.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void ld4(const double* __restrict__ p, double (&v)[4]) {
  const double2 a = __ldg(reinterpret_cast<const double2*>(p));
  const double2 b = __ldg(reinterpret_cast<const double2*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ uint32_t nibble_to_word(uint32_t nib, int lane) {
  uint32_t w = nib << (4 * (lane & 7));
  w |= __shfl_xor_sync(0xffffffffu, w, 1);
  w |= __shfl_xor_sync(0xffffffffu, w, 2);
  w |= __shfl_xor_sync(0xffffffffu, w, 4);
  return w;   // identical in the 8 lanes of a group
}

template <int G>
__global__ void __launch_bounds__(ST)
k_sets_pass1_v4(long long count, GridSpec gs, const double* __restrict__ mean, const double* __restrict__ var,
                double beta, int rule, int strict, uint32_t* __restrict__ safe_w, uint32_t* __restrict__ unsafe_w,
                SetsPartial* __restrict__ part) {
  const int lane = threadIdx.x & 31;
  ArgVal u{INFINITY, SBO_IDX_NONE}, l{INFINITY, SBO_IDX_NONE};
  long long ns = 0, nu = 0;
  for (long long base = (long long)blockIdx.x * (4 * ST); base < count; base += (long long)gridDim.x * (4 * ST)) {
    const long long p = base + 4 * threadIdx.x;
    uint32_t sb = 0, ub = 0;
    if (p < count) {
      double m[G][4], v[G][4];
#pragma unroll
      for (int i = 0; i < G; ++i) { ld4(mean + (size_t)i * count + p, m[i]); ld4(var + (size_t)i * count + p, v[i]); }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        bool safe = true, all_le = true, any_lt = false;
#pragma unroll
        for (int i = 1; i < G; ++i) {
          const double lcb = lcb_of(m[i][j], v[i][j], beta);                                  // SafeOpt.py:40-45
          safe = safe && (strict ? (lcb > 0.0) : (lcb >= 0.0));
          all_le = all_le && (lcb <= 0.0);
          any_lt = any_lt || (lcb < 0.0);
        }
        const bool unsafe = (G > 1) && (rule == SBO_UNSAFE_ALL ? all_le : any_lt);
        if (safe) {
          const long long gi = shard_global(gs, p + j);
          u = argmin2(u, ArgVal{ucb_of(m[0][j], v[0][j], beta), gi});
          l = argmin2(l, ArgVal{lcb_of(m[0][j], v[0][j], beta), gi});
          sb |= 1u << j; ++ns;
        }
        if (unsafe) { ub |= 1u << j; ++nu; }
      }
    }
    const uint32_t ws = nibble_to_word(sb, lane), wu = nibble_to_word(ub, lane);
    if ((lane & 7) == 0 && p < count) { safe_w[p >> 5] = ws; unsafe_w[p >> 5] = wu; }
  }
  // one shared-memory exchange for the four block reductions (a single barrier instead of eight: the reductions are the
  // serial tail of a bandwidth-bound CTA)
  __shared__ ArgVal sm_u[ST / 32], sm_l[ST / 32];
  __shared__ long long sm_s[ST / 32], sm_n[ST / 32];
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) {
    u = argmin2(u, shfl_xor_argval(u, m));
    l = argmin2(l, shfl_xor_argval(l, m));
    ns += __shfl_xor_sync(0xffffffffu, ns, m);
    nu += __shfl_xor_sync(0xffffffffu, nu, m);
  }
  if (lane == 0) { sm_u[threadIdx.x >> 5] = u; sm_l[threadIdx.x >> 5] = l; sm_s[threadIdx.x >> 5] = ns; sm_n[threadIdx.x >> 5] = nu; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < ST / 32; ++w) { u = argmin2(u, sm_u[w]); l = argmin2(l, sm_l[w]); ns += sm_s[w]; nu += sm_n[w]; }
    part[blockIdx.x] = SetsPartial{u.v, u.i, l.v, l.i, ns, nu};
  }
}

__global__ void __launch_bounds__(ST)
k_sets_pass2_v4(long long count, GridSpec gs, const double* __restrict__ mean, const double* __restrict__ var,
                double beta, double min_ucb0, const uint32_t* __restrict__ safe_w, uint32_t* __restrict__ min_w,
                Pass2Partial* __restrict__ part) {
  __shared__ ArgVal sm_av[ST / 32];
  __shared__ long long sm_ll[ST / 32];
  const int lane = threadIdx.x & 31;
  ArgVal a{-INFINITY, SBO_IDX_NONE};
  long long nm = 0;
  for (long long base = (long long)blockIdx.x * (4 * ST); base < count; base += (long long)gridDim.x * (4 * ST)) {
    const long long p = base + 4 * threadIdx.x;
    uint32_t mb = 0;
    if (p < count) {
      const uint32_t sb = (safe_w[p >> 5] >> (p & 31)) & 0xfu;
      if (sb) {                                      // the objective's arrays are read only where a point is safe
        double m[4], v[4];
        ld4(mean + p, m); ld4(var + p, v);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (((sb >> j) & 1u) && lcb_of(m[j], v[j], beta) <= min_ucb0) {        // SafeOpt.py:62
            mb |= 1u << j; ++nm;
            a = argmax2(a, ArgVal{v[j], shard_global(gs, p + j)});               // SafeOpt.py:55,65
          }
      }
    }
    const uint32_t wm = nibble_to_word(mb, lane);
    if ((lane & 7) == 0 && p < count) min_w[p >> 5] = wm;
  }
  a = block_argmax(a, sm_av);
  nm = block_sum_ll(nm, sm_ll);
  if (threadIdx.x == 0) part[blockIdx.x] = Pass2Partial{a.v, a.i, nm};
}

__global__ void __launch_bounds__(ST) k_sets_final2(const Pass2Partial* __restrict__ part, int nblocks, SetsDeviceResult* __restrict__ res) {
  __shared__ ArgVal sm_av[ST / 32];
  __shared__ long long sm_ll[ST / 32];
  ArgVal a{-INFINITY, SBO_IDX_NONE};
  long long nm = 0;
  for (int b = threadIdx.x; b < nblocks; b += ST) {
    a = argmax2(a, ArgVal{part[b].max_var, part[b].max_var_i});
    nm += part[b].n_min;
  }
  a = block_argmax(a, sm_av);
  nm = block_sum_ll(nm, sm_ll);
  if (threadIdx.x == 0) {
    res->max_var = a.v; res->max_var_i = (a.i == SBO_IDX_NONE) ? -1 : a.i;
    res->n_min = nm;
  }
}

// generic masked arg-reduction
struct RedPartial { double v; long long i; };
template <int KIND>
__global__ void __launch_bounds__(ST)
k_argreduce(GridSpec gs, const double* __restrict__ mean, const double* __restrict__ var, double beta,
            const uint32_t* __restrict__ mask, double t0, double t1, double t2, double t3, double t4, double t5,
            double t6, double t7, RedPartial* __restrict__ part) {
  __shared__ ArgVal sm_av[ST / 32];
  const long long count = gs.count;
  const long long p = (long long)blockIdx.x * ST + threadIdx.x;
  constexpr bool IS_MAX = (KIND == SBO_ARGMAX_VAR0);
  ArgVal a{IS_MAX ? -INFINITY : INFINITY, SBO_IDX_NONE};
  if (p < count && ((mask[p >> 5] >> (p & 31)) & 1u)) {
    double v;
    if (KIND == SBO_ARGMAX_VAR0) v = var[p];
    else if (KIND == SBO_ARGMIN_LCB0) v = lcb_of(mean[p], var[p], beta);
    else if (KIND == SBO_ARGMIN_UCB0) v = ucb_of(mean[p], var[p], beta);
    else {
      double x[SBO_MAX_D];
      point_coords(gs, shard_global(gs, p), x);
      const double t[SBO_MAX_D] = {t0, t1, t2, t3, t4, t5, t6, t7};
      v = 0.0;
      for (int k = 0; k < gs.d; ++k) { const double df = x[k] - t[k]; v = __dadd_rn(v, __dmul_rn(df, df)); }   // squared distance; sqrt on host
    }
    a = ArgVal{v, shard_global(gs, p)};
  }
  a = IS_MAX ? block_argmax(a, sm_av) : block_argmin(a, sm_av);
  if (threadIdx.x == 0) part[blockIdx.x] = RedPartial{a.v, a.i};
}
__global__ void __launch_bounds__(ST) k_argreduce_final(const RedPartial* __restrict__ part, int nblocks, int is_max,
                                                        RedPartial* __restrict__ res) {
  __shared__ ArgVal sm_av[ST / 32];
  ArgVal a{is_max ? -INFINITY : INFINITY, SBO_IDX_NONE};
  for (int b = threadIdx.x; b < nblocks; b += ST) {
    const ArgVal q{part[b].v, part[b].i};
    a = is_max ? argmax2(a, q) : argmin2(a, q);
  }
  a = is_max ? block_argmax(a, sm_av) : block_argmin(a, sm_av);
  if (threadIdx.x == 0) { res->v = a.v; res->i = (a.i == SBO_IDX_NONE) ? -1 : a.i; }
}

// ---------------------------------------------------------------------------------------------
// StableOpt on the grid (SURVEY.md section 8f row 4; models/StableOpt.py:96-160 of the reference).  The GP input is
// (x_c, d): controlled axes first (fastest), disturbance axes last, so grid point p = q + Nxc*j with q the x_c index
// and j the disturbance index.  One thread per x_c walks its disturbance column:
//   robust safe  R = {q : min_j lcb_i(q,j) >= 0 for every constraint i}        (Minimise_d(lcb, xc, i) >= 0, :147-149)
//   score(q)     = max_j fun_0(q,j),  fun = mean | ucb | lcb                   (Maximise_d(fun, xc, 0), :151)
// and the outer DE of Minimize_Maximise (:153) becomes a masked arg-min of score over R (lowest index on ties).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(ST)
k_stable_columns(int G, long long N, long long Nxc, long long Nd, const double* __restrict__ mean, const double* __restrict__ var,
                 double beta, int fun_kind, double* __restrict__ score, uint32_t* __restrict__ robust_w, RedPartial* __restrict__ part) {
  __shared__ ArgVal sm_av[ST / 32];
  const long long q = (long long)blockIdx.x * ST + threadIdx.x;
  bool safe = false;
  ArgVal a{INFINITY, SBO_IDX_NONE};
  if (q < Nxc) {
    double worst[SBO_MAX_G];
    for (int i = 1; i < G; ++i) worst[i] = INFINITY;
    double best = -INFINITY;
    for (long long j = 0; j < Nd; ++j) {
      const long long p = q + Nxc * j;
      const double m0 = mean[p], v0 = var[p];
      const double f = fun_kind == 0 ? m0 : (fun_kind == 1 ? ucb_of(m0, v0, beta) : lcb_of(m0, v0, beta));
      best = fmax(best, f);
      for (int i = 1; i < G; ++i) worst[i] = fmin(worst[i], lcb_of(mean[(size_t)i * N + p], var[(size_t)i * N + p], beta));
    }
    safe = true;
    for (int i = 1; i < G; ++i) safe = safe && (worst[i] >= 0.0);
    score[q] = best;
    if (safe) a = ArgVal{best, q};
  }
  const uint32_t w = __ballot_sync(0xffffffffu, safe);
  if ((threadIdx.x & 31) == 0 && q < Nxc) robust_w[q >> 5] = w;
  a = block_argmin(a, sm_av);
  if (threadIdx.x == 0) part[blockIdx.x] = RedPartial{a.v, a.i};
}
__global__ void __launch_bounds__(256) k_popcount_words(const uint32_t* __restrict__ w, long long nw, unsigned long long* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned c = (i < nw) ? __popc(w[i]) : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, (unsigned long long)c);
}

// ---------------------------------------------------------------------------------------------
// stream compaction of a bitmask into ascending LOCAL indices
// ---------------------------------------------------------------------------------------------
#define SC_WORDS 1024   // words per scan block
__global__ void __launch_bounds__(256) k_scan_blocksum(const uint32_t* __restrict__ mask, long long nwords, long long count,
                                                       long long* __restrict__ bsum) {
  __shared__ long long sm_ll[8];
  const long long w0 = (long long)blockIdx.x * SC_WORDS;
  long long s = 0;
  for (int t = threadIdx.x; t < SC_WORDS; t += 256) {
    const long long w = w0 + t;
    if (w < nwords) {
      uint32_t m = mask[w];
      const long long rem = count - w * 32;
      if (rem < 32) m &= (rem <= 0) ? 0u : ((1u << rem) - 1u);
      s += __popc(m);
    }
  }
  s = block_sum_ll(s, sm_ll);
  if (threadIdx.x == 0) bsum[blockIdx.x] = s;
}
// exclusive scan of the block sums by ONE CTA: every thread scans a contiguous run, the run totals are scanned
// with warp shuffles (nblocks is count/32768: 512 at C5, so one CTA is enough)
__global__ void __launch_bounds__(1024) k_scan_blocks(long long* __restrict__ bsum, int nblocks, long long* __restrict__ total) {
  __shared__ long long wsum[32];
  const int per = (nblocks + 1023) / 1024;
  const int b0 = threadIdx.x * per, b1 = min(nblocks, b0 + per);
  long long s = 0;
  for (int b = b0; b < b1; ++b) s += bsum[b];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    long long w = wsum[lane], wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += y; }
    wsum[lane] = wi - w;
    if (lane == 31) *total = wi;
  }
  __syncthreads();
  long long run = wsum[warp] + incl - s;
  for (int b = b0; b < b1; ++b) { const long long v = bsum[b]; bsum[b] = run; run += v; }
}
__global__ void __launch_bounds__(32) k_scan_scatter(const uint32_t* __restrict__ mask, long long nwords, long long count,
                                                     const long long* __restrict__ boff, long long* __restrict__ out) {
  // one warp per scan block: sequential over 32-word groups, warp-level exclusive scan of popcounts
  const long long w0 = (long long)blockIdx.x * SC_WORDS;
  long long base = boff[blockIdx.x];
  const int lane = threadIdx.x;
  for (int t = 0; t < SC_WORDS; t += 32) {
    const long long w = w0 + t + lane;
    uint32_t m = 0;
    if (w < nwords) {
      m = mask[w];
      const long long rem = count - w * 32;
      if (rem < 32) m &= (rem <= 0) ? 0u : ((1u << rem) - 1u);
    }
    const int c = __popc(m);
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
    long long pos = base + incl - c;
    while (m) { const int b = __ffs(m) - 1; m &= m - 1; out[pos++] = w * 32 + b; }
    base += __shfl_sync(0xffffffffu, incl, 31);
  }
}

int compact_mask(sbo_ctx* ctx, const uint32_t* mask_dev, long long count, DevBuf& out_idx, long long* n_out) {
  const long long nwords = cdiv(count, 32);
  const int nblocks = (int)cdiv(nwords, SC_WORDS);
  SBO_TRY(sbo_ensure(ctx, ctx->scan_a, sizeof(long long) * (nblocks + 1)));
  long long* bsum = (long long*)ctx->scan_a.p;
  k_scan_blocksum<<<nblocks, 256, 0, ctx->stream>>>(mask_dev, nwords, count, bsum);
  SBO_LAUNCH_CHECK();
  k_scan_blocks<<<1, 1024, 0, ctx->stream>>>(bsum, nblocks, bsum + nblocks);
  SBO_LAUNCH_CHECK();
  long long total = 0;
  SBO_CUDA(cudaMemcpyAsync(&total, bsum + nblocks, sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  SBO_TRY(sbo_ensure(ctx, out_idx, sizeof(long long) * (size_t)(total > 0 ? total : 1)));
  if (total > 0) {
    k_scan_scatter<<<nblocks, 32, 0, ctx->stream>>>(mask_dev, nwords, count, bsum, (long long*)out_idx.p);
    SBO_LAUNCH_CHECK();
  }
  *n_out = total;
  return SBO_OK;
}

// ---------------------------------------------------------------------------------------------
// host drivers
// ---------------------------------------------------------------------------------------------
long long mask_words(const sbo_ctx* ctx) { return cdiv(ctx->gs.count, 32); }

uint32_t* mask_ptr(sbo_ctx* ctx, int mask_kind, int which) {
  const long long nw = mask_words(ctx);
  switch (mask_kind) {
    case SBO_MASK_SAFE: return (uint32_t*)ctx->m_safe.p;
    case SBO_MASK_MIN: return (uint32_t*)ctx->m_min.p;
    case SBO_MASK_UNSAFE: return (uint32_t*)ctx->m_unsafe.p;
    case SBO_MASK_USER: return (uint32_t*)ctx->m_user.p;
    case SBO_MASK_EXPANDER: return ctx->m_exp.p ? (uint32_t*)ctx->m_exp.p + (size_t)which * nw : nullptr;
    case SBO_MASK_TARGET: return ctx->m_tgt.p ? (uint32_t*)ctx->m_tgt.p + (size_t)which * nw : nullptr;
  }
  return nullptr;
}

// persistent grid of the vectorised set kernels: 8 CTAs of 256 threads per SM (one wave), never more CTAs than tiles.
// (One tile per CTA, 2048 CTAs at the C5 shard size, measured slower: 48.4 vs 41.9 us under ncu.)
static int sets_grid(sbo_ctx* ctx, long long count) {
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  const long long tiles = cdiv(count, 4 * ST);
  return (int)(tiles < (long long)sms * 8 ? tiles : (long long)sms * 8);
}

static void fill_result(const SetsDeviceResult& r, sbo_sets_result* out) {
  out->n_safe = r.n_safe; out->n_unsafe = r.n_unsafe; out->n_min = r.n_min;
  out->min_ucb0 = r.min_ucb; out->min_ucb0_idx = r.min_ucb_i;
  out->min_lcb0 = r.min_lcb; out->min_lcb0_idx = r.min_lcb_i;
  out->minimizer_var = r.max_var; out->minimizer_idx = r.max_var_i;
}

int sets_pass1(sbo_ctx* ctx, double beta, int rule, int strict, sbo_sets_result* out) {
  SBO_REQUIRE(ctx->have_post, "sbo_sets: no posterior (call sbo_posterior)");
  SBO_REQUIRE(rule == SBO_UNSAFE_ALL || rule == SBO_UNSAFE_ANY, "bad unsafe rule");
  const long long count = ctx->gs.count;
  const long long nw = mask_words(ctx);
  const bool vec = (count % 4 == 0);
  const int nblocks = vec ? sets_grid(ctx, count) : (int)cdiv(count, ST);
  SBO_TRY(sbo_ensure(ctx, ctx->m_safe, sizeof(uint32_t) * nw));
  SBO_TRY(sbo_ensure(ctx, ctx->m_unsafe, sizeof(uint32_t) * nw));
  SBO_TRY(sbo_ensure(ctx, ctx->m_min, sizeof(uint32_t) * nw));
  SBO_TRY(sbo_ensure(ctx, ctx->partials, sizeof(SetsPartial) * (size_t)nblocks));
  SBO_TRY(sbo_ensure(ctx, ctx->result, sizeof(SetsDeviceResult) + sizeof(RedPartial)));
  ev_reset(ctx, 3);
  ev_begin(ctx, 3);
  SBO_CUDA(cudaMemsetAsync(ctx->result.p, 0, sizeof(SetsDeviceResult), ctx->stream));
  if (vec)
    with_int<1, SBO_MAX_G>(ctx->ms.G, [&](auto G) {
      k_sets_pass1_v4<G><<<nblocks, ST, 0, ctx->stream>>>(count, ctx->gs, (const double*)ctx->mean.p, (const double*)ctx->var.p,
                                                          beta, rule, strict, (uint32_t*)ctx->m_safe.p, (uint32_t*)ctx->m_unsafe.p,
                                                          (SetsPartial*)ctx->partials.p);
    });
  else
    k_sets_pass1<<<nblocks, ST, 0, ctx->stream>>>(ctx->ms.G, count, ctx->gs, (const double*)ctx->mean.p,
                                                  (const double*)ctx->var.p, beta, rule, strict,
                                                  (uint32_t*)ctx->m_safe.p, (uint32_t*)ctx->m_unsafe.p,
                                                  (SetsPartial*)ctx->partials.p);
  SBO_LAUNCH_CHECK();
  k_sets_final1<<<1, ST, 0, ctx->stream>>>((const SetsPartial*)ctx->partials.p, nblocks, (SetsDeviceResult*)ctx->result.p);
  SBO_LAUNCH_CHECK();
  ev_end(ctx);
  SetsDeviceResult r;
  SBO_CUDA(cudaMemcpyAsync(&r, ctx->result.p, sizeof(r), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  ev_collect(ctx);
  r.max_var = -INFINITY; r.max_var_i = -1; r.n_min = 0;
  if (out) fill_result(r, out);
  ctx->n_unsafe_local = r.n_unsafe;
  ctx->n_safe_local = r.n_safe;
  ctx->beta = beta;
  stage_changed(ctx, Change::SETS1);
  return SBO_OK;
}

int sets_pass2(sbo_ctx* ctx, double min_ucb0, sbo_sets_result* out) {
  SBO_REQUIRE(ctx->have_sets, "sbo_sets_pass2: call sbo_sets_pass1 first");
  const long long count = ctx->gs.count;
  const bool vec = (count % 4 == 0);
  const int nblocks = vec ? sets_grid(ctx, count) : (int)cdiv(count, ST);
  SBO_TRY(sbo_ensure(ctx, ctx->partials, sizeof(SetsPartial) * (size_t)nblocks));   // >= Pass2Partial
  ev_begin(ctx, 3);
  if (vec)
    k_sets_pass2_v4<<<nblocks, ST, 0, ctx->stream>>>(count, ctx->gs, (const double*)ctx->mean.p, (const double*)ctx->var.p,
                                                     ctx->beta, min_ucb0, (const uint32_t*)ctx->m_safe.p,
                                                     (uint32_t*)ctx->m_min.p, (Pass2Partial*)ctx->partials.p);
  else
  k_sets_pass2<<<nblocks, ST, 0, ctx->stream>>>(count, ctx->gs, (const double*)ctx->mean.p, (const double*)ctx->var.p,
                                                ctx->beta, min_ucb0, (const uint32_t*)ctx->m_safe.p,
                                                (uint32_t*)ctx->m_min.p, (Pass2Partial*)ctx->partials.p);
  SBO_LAUNCH_CHECK();
  k_sets_final2<<<1, ST, 0, ctx->stream>>>((const Pass2Partial*)ctx->partials.p, nblocks, (SetsDeviceResult*)ctx->result.p);
  SBO_LAUNCH_CHECK();
  ev_end(ctx);
  SetsDeviceResult r;
  SBO_CUDA(cudaMemcpyAsync(&r, ctx->result.p, sizeof(r), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  ev_collect(ctx);
  if (out) fill_result(r, out);
  stage_changed(ctx, Change::SETS2);
  return SBO_OK;
}

int argreduce_run(sbo_ctx* ctx, int kind, const uint32_t* mask_dev, const double* target, int64_t* idx, double* value) {
  SBO_REQUIRE(ctx->have_post, "sbo_argreduce: no posterior");
  SBO_REQUIRE(mask_dev != nullptr, "sbo_argreduce: mask not available");
  SBO_REQUIRE(kind >= 0 && kind <= 3, "bad reduce kind");
  SBO_REQUIRE(kind != SBO_ARGMIN_DIST || target != nullptr, "target required");
  const long long count = ctx->gs.count;
  const int nblocks = (int)cdiv(count, ST);
  SBO_TRY(sbo_ensure(ctx, ctx->partials, sizeof(SetsPartial) * (size_t)nblocks));
  SBO_TRY(sbo_ensure(ctx, ctx->result, sizeof(SetsDeviceResult) + sizeof(RedPartial)));
  RedPartial* part = (RedPartial*)ctx->partials.p;
  RedPartial* res = (RedPartial*)((char*)ctx->result.p + sizeof(SetsDeviceResult));
  double t[SBO_MAX_D] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (target) for (int k = 0; k < ctx->gs.d; ++k) t[k] = target[k];
  const double* mean = (const double*)ctx->mean.p;
  const double* var = (const double*)ctx->var.p;
  ev_reset(ctx, 5);
  ev_begin(ctx, 5);
  with_int<SBO_ARGMAX_VAR0, SBO_ARGMIN_DIST>(kind, [&](auto K) {
    k_argreduce<K><<<nblocks, ST, 0, ctx->stream>>>(ctx->gs, mean, var, ctx->beta, mask_dev, t[0], t[1], t[2], t[3], t[4], t[5], t[6],
                                                    t[7], part);
  });
  SBO_LAUNCH_CHECK();
  k_argreduce_final<<<1, ST, 0, ctx->stream>>>(part, nblocks, kind == SBO_ARGMAX_VAR0 ? 1 : 0, res);
  SBO_LAUNCH_CHECK();
  ev_end(ctx);
  RedPartial r;
  SBO_CUDA(cudaMemcpyAsync(&r, res, sizeof(r), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  ev_collect(ctx);
  if (idx) *idx = r.i;
  if (value) *value = (kind == SBO_ARGMIN_DIST && r.i >= 0) ? sqrt(r.v) : r.v;
  return SBO_OK;
}

// user mask = (mask_kind) AND ball ||x - x0||_2 <= r, built on the device from the implicit coordinates
// (GP_TR.BO.minimize_obj_lcb, models/GP_TR.py:43-54 of the reference: the safe set inside the trust region)
__global__ void __launch_bounds__(ST)
k_ball_mask(GridSpec gs, const uint32_t* __restrict__ src, double x0, double x1, double x2, double x3, double x4, double x5,
            double x6, double x7, double r, uint32_t* __restrict__ out) {
  const long long p = (long long)blockIdx.x * ST + threadIdx.x;
  bool in = false;
  if (p < gs.count && (!src || ((src[p >> 5] >> (p & 31)) & 1u))) {
    double x[SBO_MAX_D];
    point_coords(gs, shard_global(gs, p), x);
    const double c[SBO_MAX_D] = {x0, x1, x2, x3, x4, x5, x6, x7};
    double s = 0.0;
    for (int k = 0; k < gs.d; ++k) { const double df = __dsub_rn(x[k], c[k]); s = __dadd_rn(s, __dmul_rn(df, df)); }
    in = sqrt(s) <= r;                                  // numpy.linalg.norm(x - x0) <= r, same operations
  }
  const uint32_t w = __ballot_sync(0xffffffffu, in);
  if ((threadIdx.x & 31) == 0 && p < gs.count) out[p >> 5] = w;
}
int ball_mask(sbo_ctx* ctx, int mask_kind, const double* x0, double r) {
  SBO_REQUIRE(ctx->have_grid && x0, "sbo_user_mask_ball: no grid");
  const uint32_t* src = nullptr;
  if (mask_kind >= 0) {
    SBO_REQUIRE(ctx->have_sets, "sbo_user_mask_ball: no sets to intersect with");
    src = mask_ptr(ctx, mask_kind, 0);
    SBO_REQUIRE(src != nullptr, "mask not available");
  }
  SBO_TRY(sbo_ensure(ctx, ctx->m_user, sizeof(uint32_t) * mask_words(ctx)));
  double c[SBO_MAX_D] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int k = 0; k < ctx->gs.d; ++k) c[k] = x0[k];
  k_ball_mask<<<(unsigned)cdiv(ctx->gs.count, ST), ST, 0, ctx->stream>>>(ctx->gs, src, c[0], c[1], c[2], c[3], c[4], c[5], c[6], c[7], r,
                                                                        (uint32_t*)ctx->m_user.p);
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

// StableOpt: robust safe set + min-max over the disturbance axes of the meshgrid (see k_stable_columns)
int stable_minmax(sbo_ctx* ctx, int n_controlled, int fun_kind, double beta, int64_t* xc_idx, double* value, int64_t* n_robust_safe,
                  double* score_host) {
  SBO_REQUIRE(ctx->have_post, "sbo_stable_minmax: no posterior (call sbo_posterior)");
  const GridSpec& gs = ctx->gs;
  SBO_REQUIRE(gs.kind == 1 && gs.cyc_n <= 1 && gs.first == 0 && gs.count == gs.N, "sbo_stable_minmax needs the whole meshgrid on this context");
  SBO_REQUIRE(n_controlled >= 1 && n_controlled < gs.d, "controlled dimensions must be 1 .. d-1 (the rest are disturbances)");
  SBO_REQUIRE(fun_kind >= 0 && fun_kind <= 2, "fun_kind: 0 mean, 1 ucb, 2 lcb");
  long long Nxc = 1;
  for (int k = 0; k < n_controlled; ++k) Nxc *= gs.pts[k];
  const long long Nd = gs.N / Nxc;
  const int nblocks = (int)cdiv(Nxc, ST);
  SBO_TRY(sbo_ensure(ctx, ctx->st_score, sizeof(double) * (size_t)Nxc));
  SBO_TRY(sbo_ensure(ctx, ctx->st_mask, sizeof(uint32_t) * (size_t)cdiv(Nxc, 32)));
  SBO_TRY(sbo_ensure(ctx, ctx->partials, sizeof(SetsPartial) * (size_t)nblocks));
  SBO_TRY(sbo_ensure(ctx, ctx->result, sizeof(SetsDeviceResult) + sizeof(RedPartial)));
  RedPartial* part = (RedPartial*)ctx->partials.p;
  RedPartial* res = (RedPartial*)((char*)ctx->result.p + sizeof(SetsDeviceResult));
  SBO_TRY(sbo_ensure(ctx, ctx->pairctr, 2 * sizeof(unsigned long long)));
  unsigned long long* cnt = (unsigned long long*)ctx->pairctr.p;
  SBO_CUDA(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), ctx->stream));
  ev_reset(ctx, 3);
  ev_begin(ctx, 3);
  k_stable_columns<<<nblocks, ST, 0, ctx->stream>>>(ctx->ms.G, gs.N, Nxc, Nd, (const double*)ctx->mean.p, (const double*)ctx->var.p, beta,
                                                   fun_kind, (double*)ctx->st_score.p, (uint32_t*)ctx->st_mask.p, part);
  SBO_LAUNCH_CHECK();
  k_argreduce_final<<<1, ST, 0, ctx->stream>>>(part, nblocks, 0, res);
  SBO_LAUNCH_CHECK();
  k_popcount_words<<<(unsigned)cdiv(cdiv(Nxc, 32), 256), 256, 0, ctx->stream>>>((const uint32_t*)ctx->st_mask.p, cdiv(Nxc, 32), cnt);
  SBO_LAUNCH_CHECK();
  ev_end(ctx);
  RedPartial r;
  unsigned long long c = 0;
  SBO_CUDA(cudaMemcpyAsync(&r, res, sizeof(r), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaMemcpyAsync(&c, cnt, sizeof(c), cudaMemcpyDeviceToHost, ctx->stream));
  if (score_host) SBO_CUDA(cudaMemcpyAsync(score_host, ctx->st_score.p, sizeof(double) * (size_t)Nxc, cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  ev_collect(ctx);
  if (xc_idx) *xc_idx = r.i;
  if (value) *value = r.v;
  if (n_robust_safe) *n_robust_safe = (int64_t)c;
  return SBO_OK;
}
