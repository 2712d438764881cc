// pairs.cu -- expander / GoOSE-target pair kernels and their staged host driver.
//   Lipschitz mode (reference-exact):  ucb_idx(x) - L*||x - z + 1e-8||_2 >= 0, x in S, z in Z
//       models/SafeOpt.py:85-124 (Expander), models/GoOSE.py:69-114 (Target)
//   Fantasy mode (north_star; SURVEY.md section 8 row a12):
//       c_i = k_i(z,x) - v_z.v_x ; rank-1 update of every constraint GP with y_i = ucb_i(x);
//       z newly safe iff every updated lcb_i(z) >= 0 ; g(x) = #newly safe z.
//       FP64 SIMT reference kernel here; the TF32 tcgen05/TMEM GEMM lives in fantasy_tc.cu.
//
// Host driver in five stages so that the SAME code serves one GPU and a sharded grid (SURVEY.md 8e):
//   prepare : compact S and Z of the local shard, build the local Z-side payload
//   export  : write the local candidates' rows (coords, ucb, normalised coords, a, b) [+ V rows] to a buffer
//   import  : take the rows of ALL candidates (the all-gathered exports; on one GPU: its own export)
//   run     : pair ALL candidates with the LOCAL unsafe points -> per-candidate hit flags / newly-safe counts
//   finish  : (after the caller all-reduced the per-candidate results) masks + arg-reductions on the local shard
#include "common.cuh"
#include <math.h>
#include <string.h>

#define PT 256   // threads per pair CTA = tile length of the staged side

struct PairConsts {
  int nc;                       // number of constraints G-1
  double L[SBO_MAX_G];          // L[c] for constraint c+1
  double beta;
};

__device__ __forceinline__ bool reach_test(double s, double r2, double u, double L) {
  // exact reference predicate  u - L*sqrt(s) >= 0  (SafeOpt.py:85-88); the squared compare only
  // short-cuts pairs that are far (1e-12 relative) from the threshold.
  if (s <= r2 * (1.0 - 1e-12)) return true;
  if (s > r2 * (1.0 + 1e-12)) return false;
  return __dsub_rn(u, __dmul_rn(L, sqrt(s))) >= 0.0;
}

// ---------------------------------------------------------------------------------------------
// Exact tile culling.  bb = [lo[D][ntiles] | hi[D][ntiles] | r2max[nc][ntiles]] of the STAGED side's tiles of PT
// consecutive (grid-ordered, hence spatially compact) points.  For a fixed thread point p the reference's difference
// df_k = fl(fl(x_k - z_k) + 1e-8) is monotone in the staged coordinate, so over the tile it lies in [a_k, b_k] with
// a_k, b_k the same expression at the box corners; |df_k| >= dk = 0 if a_k <= 0 <= b_k else min(|a_k|, |b_k|), and
// because rounding is monotone the sum below (same operations, same order as the pair loop) is a lower bound of
// every pair's computed s.  reach_test(s, r2, ..) is false for every s > r2*(1+1e-12), so a tile whose lower bound
// exceeds that for every open constraint of every thread is skipped without changing any result.
// STAGED_IS_X: the thread holds z and the tile holds x (GoOSE target); otherwise the thread holds x (expander).
// ---------------------------------------------------------------------------------------------
template <int D, bool STAGED_IS_X>
__device__ __forceinline__ double tile_lower_bound(const double (&p)[D], const double* __restrict__ bb, long long ntiles, long long tile) {
  double s = 0.0;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    const double lo = bb[(size_t)k * ntiles + tile], hi = bb[(size_t)(D + k) * ntiles + tile];
    double a, b;
    if (STAGED_IS_X) {   // df = (x - z) + 1e-8, x in [lo, hi], z = p
      a = __dadd_rn(__dsub_rn(lo, p[k]), SBO_PAIR_OFFSET); b = __dadd_rn(__dsub_rn(hi, p[k]), SBO_PAIR_OFFSET);
    } else {             // x = p, z in [lo, hi]
      a = __dadd_rn(__dsub_rn(p[k], hi), SBO_PAIR_OFFSET); b = __dadd_rn(__dsub_rn(p[k], lo), SBO_PAIR_OFFSET);
    }
    const double dk = (a <= 0.0 && b >= 0.0) ? 0.0 : fmin(fabs(a), fabs(b));
    s = __dadd_rn(s, __dmul_rn(dk, dk));
  }
  return s;
}

// bounding boxes (and, with thr, the largest radius^2 per constraint) of tiles of PT consecutive points
template <int D>
__global__ void __launch_bounds__(PT)
k_tile_bbox(long long n, long long ntiles, const double* __restrict__ coords, int nc, const double* __restrict__ thr,
            double* __restrict__ bb) {
  __shared__ double red[PT / 32];
  const long long tile = blockIdx.x, i = tile * PT + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  auto block_reduce = [&](double v, bool want_max) -> double {
    for (int o = 16; o > 0; o >>= 1) {
      const double w = __shfl_xor_sync(0xffffffffu, v, o);
      v = want_max ? fmax(v, w) : fmin(v, w);
    }
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double r = red[0];
    for (int w = 1; w < PT / 32; ++w) r = want_max ? fmax(r, red[w]) : fmin(r, red[w]);
    return r;
  };
  for (int k = 0; k < D; ++k) {
    const double v = (i < n) ? coords[(size_t)k * n + i] : 0.0;
    const double lo = block_reduce((i < n) ? v : INFINITY, false);
    const double hi = block_reduce((i < n) ? v : -INFINITY, true);
    if (threadIdx.x == 0) { bb[(size_t)k * ntiles + tile] = lo; bb[(size_t)(D + k) * ntiles + tile] = hi; }
  }
  for (int c = 0; c < nc; ++c) {
    const double r = block_reduce((i < n && thr) ? thr[(size_t)c * n + i] : -1.0, true);
    if (threadIdx.x == 0 && thr) bb[(size_t)(2 * D + c) * ntiles + tile] = r;
  }
}

// ---------------------------------------------------------------------------------------------
// SafeOpt expander: one thread per candidate x, z tiles staged in shared memory.
// hits[c][t] = 1 if some z is reachable from x_t under constraint c+1.
// ---------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(PT)
k_pairs_expander(PairConsts pc, long long nx, long long nz, const double* __restrict__ xc, const double* __restrict__ ucb,
                 const double* __restrict__ thr, const double* __restrict__ zc, unsigned char* __restrict__ hits,
                 unsigned long long* __restrict__ pair_counter, long long z_per_split, const double* __restrict__ bb,
                 long long ntiles, int tile_stride, int tile_offset, const int* __restrict__ out_pos) {
  __shared__ double zs[D][PT];
  // candidate tiles are dealt round-robin to the ranks of a sharded run (tile_stride = nranks, tile_offset = rank)
  const long long t = ((long long)blockIdx.x * tile_stride + tile_offset) * PT + threadIdx.x;
  const bool active = t < nx;
  double x[D], u[SBO_MAX_G - 1], r2[SBO_MAX_G - 1];
  const unsigned full = (1u << pc.nc) - 1u;
  unsigned found = 0;
  if (active) {
#pragma unroll
    for (int k = 0; k < D; ++k) x[k] = xc[(size_t)k * nx + t];
    for (int c = 0; c < pc.nc; ++c) {
      u[c] = ucb[(size_t)c * nx + t]; r2[c] = thr[(size_t)c * nx + t];
    }
  } else {
    found = full;
  }
  unsigned dead = 0;   // constraints that can never hit for this x
  if (active) for (int c = 0; c < pc.nc; ++c) if (r2[c] < 0.0) dead |= 1u << c;
  const long long z0 = (long long)blockIdx.y * z_per_split;
  const long long z1 = min(nz, z0 + z_per_split);
  unsigned long long tiles = 0;
  const long long o_hit = active ? (out_pos ? (long long)out_pos[t] : t) : 0;
  int poll = 0;
  for (long long zb = z0; zb < z1; zb += PT) {
    // the z range is split over blockIdx.y: a hit found by another split settles the constraint here as well (the flags
    // are only ever set, so a stale read costs work, never correctness)
    if (gridDim.y > 1 && active && (++poll & 3) == 0)
      for (int c = 0; c < pc.nc; ++c)
        if (!((found >> c) & 1u) && *(volatile const unsigned char*)(hits + (size_t)c * nx + o_hit)) found |= 1u << c;
    if (__syncthreads_and((found | dead) == full)) break;
    if (bb) {   // exact culling: skip the tile when no thread's x can reach its bounding box (see tile_lower_bound)
      bool need = false;
      if (active && (found | dead) != full) {
        const double slb = tile_lower_bound<D, false>(x, bb, ntiles, zb / PT);
        for (int c = 0; c < pc.nc; ++c)
          if (!(((found | dead) >> c) & 1u) && slb <= r2[c] * (1.0 + 1e-12)) need = true;
      }
      if (!__syncthreads_or(need)) continue;
    }
    const long long zi = zb + threadIdx.x;
#pragma unroll
    for (int k = 0; k < D; ++k) zs[k][threadIdx.x] = (zi < z1) ? zc[(size_t)k * nz + zi] : INFINITY;
    __syncthreads();
    ++tiles;
    if (active && (found | dead) != full) {
      const int tn = (int)min((long long)PT, z1 - zb);
      for (int j = 0; j < tn; ++j) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < D; ++k) {
          const double df = __dadd_rn(__dsub_rn(x[k], zs[k][j]), SBO_PAIR_OFFSET);   // (x - z) + 1e-8, SafeOpt.py:87
          s = __dadd_rn(s, __dmul_rn(df, df));
        }
        for (int c = 0; c < pc.nc; ++c)
          if (!((found >> c) & 1u) && r2[c] >= 0.0 && reach_test(s, r2[c], u[c], pc.L[c])) {
            found |= 1u << c;
            if (gridDim.y > 1) hits[(size_t)c * nx + o_hit] = 1;       // publish at once: the other z splits stop looking
          }
      }
    }
  }
  if (active) {
    for (int c = 0; c < pc.nc; ++c)                    // hit flags go back in the caller's (gathered) candidate order
      if ((found >> c) & 1u) hits[(size_t)c * nx + o_hit] = 1;
  }
  if (threadIdx.x == 0 && pair_counter) atomicAdd(pair_counter, tiles * (unsigned long long)PT * PT * pc.nc);
}

// ---------------------------------------------------------------------------------------------
// GoOSE target: one thread per unsafe z, x tiles (coords, radius^2, ucb) staged in shared memory.
// hits[c][t] = 1 if z_t is reachable from some safe x under constraint c+1.
// ---------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(PT)
k_pairs_target(PairConsts pc, long long nx, long long nz, const double* __restrict__ xc, const double* __restrict__ ucb,
               const double* __restrict__ thr, const double* __restrict__ zc, unsigned char* __restrict__ hits,
               unsigned long long* __restrict__ pair_counter, long long x_per_split, const double* __restrict__ bb,
               long long ntiles, int tile_stride, int tile_offset) {
  __shared__ double xs[D][PT];
  __shared__ double us[SBO_MAX_G - 1][PT];
  __shared__ double rs[SBO_MAX_G - 1][PT];
  // sharded runs over the all-gathered unsafe set: z tiles are dealt round-robin to the ranks
  const long long t = ((long long)blockIdx.x * tile_stride + tile_offset) * PT + threadIdx.x;
  const bool active = t < nz;
  double z[D];
  const unsigned full = (1u << pc.nc) - 1u;
  unsigned found = active ? 0u : full;
  if (active) {
#pragma unroll
    for (int k = 0; k < D; ++k) z[k] = zc[(size_t)k * nz + t];
  }
  const long long x0 = (long long)blockIdx.y * x_per_split;
  const long long x1 = min(nx, x0 + x_per_split);
  unsigned long long tiles = 0;
  int poll = 0;
  for (long long xb = x0; xb < x1; xb += PT) {
    if (gridDim.y > 1 && active && (++poll & 3) == 0)      // a hit found by another x split settles the constraint here too
      for (int c = 0; c < pc.nc; ++c)
        if (!((found >> c) & 1u) && *(volatile const unsigned char*)(hits + (size_t)c * nz + t)) found |= 1u << c;
    if (__syncthreads_and(found == full)) break;
    if (bb) {   // exact culling against the x tile's bounding box and its largest radius per constraint
      bool need = false;
      if (active && found != full) {
        const long long tile = xb / PT;
        const double slb = tile_lower_bound<D, true>(z, bb, ntiles, tile);
        const double* r2max = bb + (size_t)2 * D * ntiles;
        for (int c = 0; c < pc.nc; ++c) {
          const double rm = r2max[(size_t)c * ntiles + tile];
          if (!((found >> c) & 1u) && rm >= 0.0 && slb <= rm * (1.0 + 1e-12)) need = true;
        }
      }
      if (!__syncthreads_or(need)) continue;
    }
    const long long xi = xb + threadIdx.x;
#pragma unroll
    for (int k = 0; k < D; ++k) xs[k][threadIdx.x] = (xi < x1) ? xc[(size_t)k * nx + xi] : INFINITY;
    for (int c = 0; c < pc.nc; ++c) {
      us[c][threadIdx.x] = (xi < x1) ? ucb[(size_t)c * nx + xi] : -1.0;
      rs[c][threadIdx.x] = (xi < x1) ? thr[(size_t)c * nx + xi] : -1.0;
    }
    __syncthreads();
    ++tiles;
    if (active && found != full) {
      const int tn = (int)min((long long)PT, x1 - xb);
      for (int j = 0; j < tn; ++j) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < D; ++k) {
          const double df = __dadd_rn(__dsub_rn(xs[k][j], z[k]), SBO_PAIR_OFFSET);   // (x - z) + 1e-8, GoOSE.py:71
          s = __dadd_rn(s, __dmul_rn(df, df));
        }
        for (int c = 0; c < pc.nc; ++c) {
          const double r2 = rs[c][j];
          if (!((found >> c) & 1u) && r2 >= 0.0 && reach_test(s, r2, us[c][j], pc.L[c])) {
            found |= 1u << c;
            if (gridDim.y > 1) hits[(size_t)c * nz + t] = 1;
          }
        }
      }
    }
  }
  if (active) {
    for (int c = 0; c < pc.nc; ++c)
      if ((found >> c) & 1u) hits[(size_t)c * nz + t] = 1;
  }
  if (threadIdx.x == 0 && pair_counter) atomicAdd(pair_counter, tiles * (unsigned long long)PT * PT * pc.nc);
}

template <int D>
static int launch_pairs(sbo_ctx* ctx, bool goose, const PairConsts& pc, long long nx, long long nz, const double* xc,
                        const double* ucb, const double* thr, const double* zc, unsigned char* hits,
                        unsigned long long* ctr, int tile_stride, int tile_offset, const int* out_pos) {
  const long long nthr = goose ? nz : nx, ntile = goose ? nx : nz;
  long long bx = cdiv(nthr, PT);
  if (tile_stride > 1) bx = bx > tile_offset ? cdiv(bx - tile_offset, tile_stride) : 0;   // this rank's share of the thread-side tiles
  if (bx == 0) return SBO_OK;
  long long splits = 1;
  const long long tiles = cdiv(ntile, PT);
  // many small work units: the cost of a CTA varies by orders of magnitude (points next to the safe-set boundary scan
  // many tiles, far ones are culled at once), so a single wave of CTAs -- a sharded run has 1/nranks of the thread-side
  // points -- leaves the GPU waiting for the slowest one.  The splits share hits through the global flags.
  while (bx * splits < 16 * 148 && splits * 8 <= tiles && splits < 65535) splits *= 2;
  const long long per = cdiv(cdiv(ntile, splits), PT) * PT;
  dim3 grid((unsigned)bx, (unsigned)cdiv(ntile, per));
  // bounding boxes of the staged side's tiles for the exact culling (option pair_cull, default on)
  double* bb = nullptr;
  if (ctx->opt_pair_cull) {
    SBO_TRY(sbo_ensure(ctx, ctx->tile_bb, sizeof(double) * (size_t)(2 * D + pc.nc) * tiles));
    bb = (double*)ctx->tile_bb.p;
    k_tile_bbox<D><<<(unsigned)tiles, PT, 0, ctx->stream>>>(ntile, tiles, goose ? xc : zc, pc.nc, goose ? thr : nullptr, bb);
    ctx->launches++;
  }
  if (goose)
    k_pairs_target<D><<<grid, PT, 0, ctx->stream>>>(pc, nx, nz, xc, ucb, thr, zc, hits, ctr, per, bb, tiles,
                                                    tile_stride > 1 ? tile_stride : 1, tile_stride > 1 ? tile_offset : 0);
  else
    k_pairs_expander<D><<<grid, PT, 0, ctx->stream>>>(pc, nx, nz, xc, ucb, thr, zc, hits, ctr, per, bb, tiles,
                                                      tile_stride > 1 ? tile_stride : 1, tile_stride > 1 ? tile_offset : 0, out_pos);
  return SBO_OK;
}

// ---------------------------------------------------------------------------------------------
// payload kernels
// ---------------------------------------------------------------------------------------------
// raw coordinates of compacted local points (SoA): coords[k][t]
__global__ void __launch_bounds__(256)
k_gather_coords(GridSpec gs, const long long* __restrict__ idx, long long n, double* __restrict__ coords) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  double x[SBO_MAX_D];
  point_coords(gs, shard_global(gs, idx[t]), x);
  for (int k = 0; k < gs.d; ++k) coords[(size_t)k * n + t] = x[k];
}

// raw coordinates of points given by GLOBAL grid index (the all-gathered unsafe set of a sharded Lipschitz expander)
__global__ void __launch_bounds__(256)
k_gather_coords_global(GridSpec gs, const long long* __restrict__ gidx, long long n, double* __restrict__ coords) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  double x[SBO_MAX_D];
  point_coords(gs, gidx[t], x);
  for (int k = 0; k < gs.d; ++k) coords[(size_t)k * n + t] = x[k];
}
// global bitmask over the whole grid from the ranks' local masks (rotated block-cyclic shards, common.cuh shard_global):
// global word w lies in block b = w*32/blk, super-block sb = b/n, slot = b%n, owner r = (slot - rot(sb)) mod n,
// where it is local word sb*(blk/32) + w%(blk/32) of that rank's mask.
__global__ void __launch_bounds__(256)
k_assemble_global_mask(long long n_words, long long blk, int nranks, const uint32_t* __restrict__ gathered,
                       long long words_per_rank, uint32_t* __restrict__ out) {
  const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_words) return;
  const long long wpb = blk / 32, b = w / wpb, sb = b / nranks, n = nranks;
  const long long slot = b % n, rot = (sb + sb / n + sb / (n * n)) % n;
  const long long r = (slot - rot + n) % n;
  const long long lw = sb * wpb + w % wpb;
  out[w] = (lw < words_per_rank) ? gathered[(size_t)r * words_per_rank + lw] : 0u;
}
// canonical (ascending global index) slot of every gathered candidate row; the rows of each rank's segment are already
// ascending, so the slot is a sum of lower bounds over the segments (deterministic on every rank)
__global__ void __launch_bounds__(256)
k_canon_perm(long long n, int nseg, const long long* __restrict__ seg_off, const double* __restrict__ rows, int RS,
             int* __restrict__ perm) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double g = rows[(size_t)i * RS + RS - 1];
  long long pos = 0;
  for (int r = 0; r < nseg; ++r) {
    long long lo = seg_off[r], hi = seg_off[r + 1];
    if (i >= lo && i < hi) { pos += i - lo; continue; }
    const long long base = lo;
    while (lo < hi) { const long long m = (lo + hi) >> 1; if (rows[(size_t)m * RS + RS - 1] < g) lo = m + 1; else hi = m; }
    pos += lo - base;
  }
  perm[pos] = (int)i;
}

// export row of one local candidate (doubles): [coords[d] | ucb[nc] | xn[d] | a[nc] | b[nc] | global grid index]
//   a = beta*sigma/(sigma^2+sn2), b = 1/(sigma^2+sn2) in normalised units (fantasy update gains)
__global__ void __launch_bounds__(256)
k_export_rows(GridSpec gs, ModelSpec ms, double beta, const long long* __restrict__ idx, long long n,
              const double* __restrict__ mean, const double* __restrict__ var, double* __restrict__ rows) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int d = gs.d, nc = ms.G - 1;
  const int RS = 2 * d + 3 * nc + 1;
  const long long p = idx[t];
  double x[SBO_MAX_D];
  point_coords(gs, shard_global(gs, p), x);
  double* r = rows + (size_t)t * RS;
  r[RS - 1] = (double)shard_global(gs, p);             // exact below 2^53
  for (int k = 0; k < d; ++k) { r[k] = x[k]; r[d + nc + k] = (x[k] - ms.Xmean[k]) / ms.Xstd[k]; }
  for (int c = 0; c < nc; ++c) {
    const double m = mean[(size_t)(c + 1) * gs.count + p], v = var[(size_t)(c + 1) * gs.count + p];
    r[d + c] = ucb_of(m, v, beta);
    const double ys = ms.Ystd[c + 1];
    const double vn = v / (ys * ys);
    const double den = vn + ms.sn2[c + 1];
    r[2 * d + nc + c] = beta * sqrt(vn) / den;
    r[2 * d + 2 * nc + c] = 1.0 / den;
  }
}

// V rows of the local candidates, candidate-major: out[t][c][rowlen]
template <typename T>
__global__ void __launch_bounds__(256)
k_export_v(int nc, int rowlen, long long n, long long vcount, const long long* __restrict__ idx,
           const T* __restrict__ vall, T* __restrict__ out) {
  const long long t = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int c = blockIdx.y;
  if (t >= n) return;
  const int lane = threadIdx.x & 31;
  const T* s = vall + ((size_t)c * vcount + idx[t]) * rowlen;
  T* o = out + ((size_t)t * nc + c) * rowlen;
  for (int k = lane; k < rowlen; k += 32) o[k] = s[k];
}

// imported rows (AoS) -> SoA payloads of the pair kernels
__global__ void __launch_bounds__(256)
k_import_rows(int d, int nc, long long n, PairConsts pc, const int* __restrict__ perm, const double* __restrict__ rows, double* __restrict__ coords,
              double* __restrict__ ucb, double* __restrict__ thr, double* __restrict__ xn, double* __restrict__ ax,
              double* __restrict__ bx) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int RS = 2 * d + 3 * nc + 1;
  const double* r = rows + (size_t)(perm ? perm[t] : t) * RS;        // slot t holds gathered candidate perm[t]
  for (int k = 0; k < d; ++k) { coords[(size_t)k * n + t] = r[k]; xn[(size_t)k * n + t] = r[d + nc + k]; }
  for (int c = 0; c < nc; ++c) {
    const double u = r[d + c];
    ucb[(size_t)c * n + t] = u;
    double r2;
    if (!(u >= 0.0)) r2 = -1.0;
    else if (pc.L[c] > 0.0) { const double q = u / pc.L[c]; r2 = q * q; }
    else r2 = INFINITY;
    thr[(size_t)c * n + t] = r2;
    ax[(size_t)c * n + t] = r[2 * d + nc + c];
    bx[(size_t)c * n + t] = r[2 * d + 2 * nc + c];
  }
}

// imported V rows [t][c][rowlen] -> GEMM operand layout Vx[c][nxp][rowlen], zero rows for t >= n
template <typename T>
__global__ void __launch_bounds__(256)
k_import_v(int nc, int rowlen, long long n, long long npadrows, const int* __restrict__ perm, const T* __restrict__ in, T* __restrict__ vout) {
  const long long t = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int c = blockIdx.y;
  if (t >= npadrows) return;
  const int lane = threadIdx.x & 31;
  T* o = vout + ((size_t)c * npadrows + t) * rowlen;
  if (t < n) {
    const T* s = in + ((size_t)(perm ? perm[t] : t) * nc + c) * rowlen;
    for (int k = lane; k < rowlen; k += 32) o[k] = s[k];
  } else {
    for (int k = lane; k < rowlen; k += 32) o[k] = (T)0;
  }
}

// gather V rows of compacted LOCAL points: Vout[c][t][0..rowlen) = vall[c][idx[t]][..]  (zero rows for padding)
template <typename T>
__global__ void __launch_bounds__(256)
k_gather_rows(int nc, int rowlen, long long n, long long npadrows, long long vcount, const long long* __restrict__ idx,
              const T* __restrict__ vall, T* __restrict__ vout) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int c = blockIdx.y;
  if (row >= npadrows) return;
  const int lane = threadIdx.x & 31;
  T* o = vout + ((size_t)c * npadrows + row) * rowlen;
  if (row < n) {
    const T* s = vall + ((size_t)c * vcount + idx[row]) * rowlen;
    for (int k = lane; k < rowlen; k += 32) o[k] = s[k];
  } else {
    for (int k = lane; k < rowlen; k += 32) o[k] = (T)0;
  }
}

// z-side auxiliaries in NORMALISED units: zn[k][t], m[c][t] = mean_raw/Ystd, s[c][t] = var_raw/Ystd^2
__global__ void __launch_bounds__(256)
k_fantasy_aux_z(GridSpec gs, ModelSpec ms, const long long* __restrict__ idx, long long n,
                const double* __restrict__ mean, const double* __restrict__ var,
                double* __restrict__ zn, double* __restrict__ m, double* __restrict__ s) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const long long p = idx[t];
  double x[SBO_MAX_D];
  point_coords(gs, shard_global(gs, p), x);
  for (int k = 0; k < gs.d; ++k) zn[(size_t)k * n + t] = (x[k] - ms.Xmean[k]) / ms.Xstd[k];
  for (int c = 0; c < ms.G - 1; ++c) {
    const double ys = ms.Ystd[c + 1];
    m[(size_t)c * n + t] = mean[(size_t)(c + 1) * gs.count + p] / ys;
    s[(size_t)c * n + t] = var[(size_t)(c + 1) * gs.count + p] / (ys * ys);
  }
}

// ---------------------------------------------------------------------------------------------
// Exact pruning of the fantasy expander (option fantasy_prune, default on).  The posterior covariance is PSD, so
// |cov_c(z,x)| <= sigma_c(x) sigma_c(z); the updated bound  f(cov) = m_z + a_x cov - beta sqrt(s_z - b_x cov^2)  satisfies
// f(-|cov|) <= f(|cov|) and is increasing for cov >= 0, hence for EVERY pair
//     lcb'_c(z | x) <= m_z + beta sigma_z q_xc ,   q_xc = kappa - sqrt(1 - kappa),  kappa = sigma_x^2/(sigma_x^2 + sn2_c).
// z can become safe through x only if  rho_zc := -m_zc/(beta sigma_zc) <= q_xc  for every constraint, which implies the
// scalar test  key_z := max_c rho_zc  <=  key_x := max_c q_xc.  Candidates and unsafe points are ordered by their keys
// (counting sort, 4096 bins), so the feasible (x tile, z tile) pairs form a staircase and every other tile pair is
// skipped without changing any count (C4: 34 % of the tile pairs remain).  key_z > 1 can never be reached (q < 1):
// those z are dropped altogether (the round-1 z-side pruning).  Slack: 1e-9 absolute on m_z (normalised units) and
// 1e-6 on key_x, far above FP64 rounding of the bound and far below anything that matters for the pruning ratio.
// ---------------------------------------------------------------------------------------------
#define SORT_BINS 4096
__device__ __forceinline__ int key_bin(double key) {
  if (!(key >= -1.0)) return 0;                       // also NaN
  if (key > 1.0) return SORT_BINS - 1;                // overflow bin: infeasible for every candidate
  const int b = 1 + (int)((key + 1.0) * 0.5 * (SORT_BINS - 2));
  return b > SORT_BINS - 2 ? SORT_BINS - 2 : b;
}
__global__ void __launch_bounds__(256)
k_key_z(int G, long long count, double beta, ModelSpec ms, const long long* __restrict__ idx, long long n,
        const double* __restrict__ mean, const double* __restrict__ var, double* __restrict__ key) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const long long p = idx[t];
  double k = -INFINITY;
  for (int i = 1; i < G; ++i) {
    const double num = -mean[(size_t)i * count + p] - 1e-9 * ms.Ystd[i];
    const double den = beta * sqrt(var[(size_t)i * count + p]);
    const double rho = (den > 0.0) ? num / den : (num > 0.0 ? INFINITY : -INFINITY);
    k = fmax(k, rho);
  }
  key[t] = k;
}
// key_x from the gathered candidate rows [coords d | ucb nc | xn d | a nc | b nc]: kappa_c = 1 - sn2_c * b_c
__global__ void __launch_bounds__(256)
k_key_x(int d, int nc, long long n, FantasyConsts fc, const double* __restrict__ rows, double* __restrict__ key) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const double* r = rows + (size_t)t * (2 * d + 3 * nc + 1);
  double k = -INFINITY;
  for (int c = 0; c < nc; ++c) {
    const double kap = fmin(fmax(1.0 - fc.sn2[c] * r[2 * d + 2 * nc + c], 0.0), 1.0);
    k = fmax(k, kap - sqrt(1.0 - kap));
  }
  key[t] = k + 1e-6;
}
__global__ void __launch_bounds__(256)
k_sort_hist(long long n, const double* __restrict__ key, int* __restrict__ hist) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) atomicAdd(hist + key_bin(key[t]), 1);
}
// one CTA: exclusive scan of the SORT_BINS counters into cursor[]; total[0] = n, total[1] = entries below the overflow bin
__global__ void __launch_bounds__(1024) k_sort_scan(const int* __restrict__ hist, int* __restrict__ cursor, long long* __restrict__ total) {
  __shared__ int wsum[32];
  constexpr int PER = SORT_BINS / 1024;
  int v[PER], s = 0;
#pragma unroll
  for (int i = 0; i < PER; ++i) { v[i] = hist[threadIdx.x * PER + i]; s += v[i]; }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = wsum[lane], wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += y; }
    wsum[lane] = wi - w;
    if (lane == 31) total[0] = wi;
  }
  __syncthreads();
  int run = wsum[warp] + incl - s;
#pragma unroll
  for (int i = 0; i < PER; ++i) { cursor[threadIdx.x * PER + i] = run; run += v[i]; }
  if (threadIdx.x == 1023) total[1] = run - v[PER - 1];     // start of the overflow bin
}
// perm[sorted slot] = original position (order inside a bin is arbitrary: no result depends on it)
__global__ void __launch_bounds__(256)
k_sort_scatter(long long n, const double* __restrict__ key, int* __restrict__ cursor, int* __restrict__ perm) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) perm[atomicAdd(cursor + key_bin(key[t]), 1)] = (int)t;
}
__global__ void __launch_bounds__(256)
k_permute_idx(long long n, const int* __restrict__ perm, const long long* __restrict__ in, long long* __restrict__ out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = in[perm[t]];
}
__global__ void __launch_bounds__(256)
k_permute_key(long long n, const int* __restrict__ perm, const double* __restrict__ in, double* __restrict__ out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = in[perm[t]];
}
// counting sort of n keys: perm_out[sorted slot] = original position; n_below = entries with key <= 1
static int sort_by_key(sbo_ctx* ctx, long long n, const double* key, DevBuf& perm_buf, long long* n_below) {
  SBO_REQUIRE(n < 2000000000LL, "too many points to sort");
  SBO_TRY(sbo_ensure(ctx, ctx->sort_ws, sizeof(int) * 2 * SORT_BINS + 2 * sizeof(long long)));
  SBO_TRY(sbo_ensure(ctx, perm_buf, sizeof(int) * (size_t)(n > 0 ? n : 1)));
  int* hist = (int*)ctx->sort_ws.p; int* cursor = hist + SORT_BINS; long long* total = (long long*)(cursor + SORT_BINS);
  SBO_CUDA(cudaMemsetAsync(hist, 0, sizeof(int) * SORT_BINS, ctx->stream));
  k_sort_hist<<<(unsigned)cdiv(n, 256), 256, 0, ctx->stream>>>(n, key, hist);
  SBO_LAUNCH_CHECK();
  k_sort_scan<<<1, 1024, 0, ctx->stream>>>(hist, cursor, total);
  SBO_LAUNCH_CHECK();
  k_sort_scatter<<<(unsigned)cdiv(n, 256), 256, 0, ctx->stream>>>(n, key, cursor, (int*)perm_buf.p);
  SBO_LAUNCH_CHECK();
  if (n_below) {
    long long h[2];
    SBO_CUDA(cudaMemcpyAsync(h, total, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    SBO_CUDA(cudaStreamSynchronize(ctx->stream));
    *n_below = h[1];
  }
  return SBO_OK;
}

// per-element results -> bitmask words of the local shard (one mask per constraint)
__global__ void __launch_bounds__(256)
k_hits_to_mask(int nc, long long n, long long stride, long long offset, const long long* __restrict__ idx,
               const unsigned char* __restrict__ hits, uint32_t* __restrict__ masks, long long nwords) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const long long p = idx[t];
  for (int c = 0; c < nc; ++c)
    if (hits[(size_t)c * stride + offset + t]) atomicOr(masks + (size_t)c * nwords + (p >> 5), 1u << (p & 31));
}
__global__ void __launch_bounds__(256)
k_counts_scatter(long long n, long long offset, const long long* __restrict__ idx, const int* __restrict__ cnt_c,
                 int* __restrict__ cnt_pt, uint32_t* __restrict__ mask) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const long long p = idx[t];
  const int c = cnt_c[offset + t];
  if (cnt_pt) cnt_pt[p] = c;
  if (c > 0) atomicOr(mask + (p >> 5), 1u << (p & 31));
}
// bounds mode: candidates the error bound leaves undecided (no settled newly-safe pair, at least one ambiguous pair)
__global__ void __launch_bounds__(256)
k_undecided_mask(long long n, long long offset, const long long* __restrict__ idx, const int* __restrict__ cnt_c,
                 const int* __restrict__ amb_c, int* __restrict__ cnt_pt, uint32_t* __restrict__ mask) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  if (cnt_c[offset + t] > 0 || amb_c[offset + t] == 0) return;
  const long long p = idx[t];
  if (cnt_pt) cnt_pt[p] = -1;
  atomicOr(mask + (p >> 5), 1u << (p & 31));
}
__global__ void __launch_bounds__(256)
k_union_count(int nc, const uint32_t* __restrict__ masks, long long nwords, unsigned long long* __restrict__ out) {
  const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned c = 0;
  if (w < nwords) {
    uint32_t m = 0;
    for (int i = 0; i < nc; ++i) m |= masks[(size_t)i * nwords + w];
    c = __popc(m);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, (unsigned long long)c);
}

// =============================================================================================
// Fantasy mode, FP64 SIMT reference kernel (rows = z, columns = x)
// =============================================================================================
#define FB 64
#define FK 16
template <int D, bool TARGET, class KC>   // TARGET: GoOSE target epilogue (column OR into hit_words); KC: covariance function
__global__ void __launch_bounds__(256)
k_fantasy_f64(FantasyConsts fc, long long nx, long long nz, long long nxp, long long nzp,
              const double* __restrict__ Vx, const double* __restrict__ Vz,
              const double* __restrict__ xn, const double* __restrict__ ax, const double* __restrict__ bx,
              const double* __restrict__ zn, const double* __restrict__ mz, const double* __restrict__ sz,
              int* __restrict__ counts, const double* __restrict__ key_x, const double* __restrict__ key_z,
              const int* __restrict__ row_perm, unsigned long long* __restrict__ pair_counter, uint32_t* __restrict__ hit_words) {
  __shared__ double As[FK][FB + 1];   // z rows
  __shared__ double Bs[FK][FB + 1];   // x rows
  __shared__ int cnt[16][FB];
  __shared__ uint32_t hw[FB / 32];    // GoOSE target: the block's z rows made safe by some valid x column
  const KC kc(fc.kernel);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const long long zb = (long long)blockIdx.x * FB, xb = (long long)blockIdx.y * FB;
  if (key_x) {   // exact pruning (see k_key_z): no pair of this block can become safe when min key_z > max key_x
    bool reach = false;
    if (tid < FB) {
      const double kx = (xb + tid < nx) ? key_x[xb + tid] : -INFINITY;
      double qm = kx;
      for (int o = 16; o > 0; o >>= 1) qm = fmax(qm, __shfl_xor_sync(0xffffffffu, qm, o));
      const double kz = (zb + tid < nz) ? key_z[zb + tid] : INFINITY;
      double rm = kz;
      for (int o = 16; o > 0; o >>= 1) rm = fmin(rm, __shfl_xor_sync(0xffffffffu, rm, o));
      As[0][tid] = qm; Bs[0][tid] = rm;
    }
    __syncthreads();
    reach = fmin(Bs[0][0], Bs[0][32]) <= fmax(As[0][0], As[0][32]);
    __syncthreads();
    if (!reach) return;
  }
  if (tid == 0 && pair_counter) atomicAdd(pair_counter, (unsigned long long)FB * FB);
  if (TARGET && tid < FB / 32) hw[tid] = 0u;
  const int np = fc.npad;
  unsigned okmask = 0xffffu;   // bit i*4+j
  double zc[4][D], xc[4][D];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long zi = zb + ty * 4 + i, xi = xb + tx * 4 + i;
#pragma unroll
    for (int k = 0; k < D; ++k) {
      zc[i][k] = (zi < nz) ? zn[(size_t)k * nz + zi] : 0.0;
      xc[i][k] = (xi < nx) ? xn[(size_t)k * nx + xi] : 0.0;
    }
  }
  for (int c = 0; c < fc.nc; ++c) {
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    const double* Az = Vz + ((size_t)c * nzp + zb) * np;
    const double* Bx = Vx + ((size_t)c * nxp + xb) * np;
    for (int k0 = 0; k0 < np; k0 += FK) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int e = tid + 256 * q;
        const int r = e >> 4, kk = e & 15;
        As[kk][r] = Az[(size_t)r * np + k0 + kk];
        Bs[kk][r] = Bx[(size_t)r * np + k0 + kk];
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < FK; ++kk) {
        double a4[4], b4[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { a4[i] = As[kk][ty * 4 + i]; b4[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fma(a4[i], b4[j], acc[i][j]);
      }
      __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long zi = zb + ty * 4 + i;
      const double m_z = (zi < nz) ? mz[(size_t)c * nz + zi] : 0.0;
      const double s_z = (zi < nz) ? sz[(size_t)c * nz + zi] : 0.0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const long long xi = xb + tx * 4 + j;
        const double a_x = (xi < nx) ? ax[(size_t)c * nx + xi] : 0.0;
        const double b_x = (xi < nx) ? bx[(size_t)c * nx + xi] : 0.0;
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < D; ++k) { const double df = zc[i][k] - xc[j][k]; s += df * df * fc.inv_ell[c][k]; }
        const double cc = kc.value(s, fc.sf2[c]) - acc[i][j];
        const double mu = m_z + cc * a_x;
        const double s2 = s_z - cc * cc * b_x;
        const bool ok = (mu - fc.beta * sqrt(fmax(s2, 0.0))) >= 0.0;
        if (!ok) okmask &= ~(1u << (i * 4 + j));
      }
    }
  }
  if (TARGET) {   // GoOSE target: OR over the valid x columns of every valid z row
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = ty * 4 + i;
      bool any = false;
#pragma unroll
      for (int j = 0; j < 4; ++j) any |= xb + tx * 4 + j < nx && ((okmask >> (i * 4 + j)) & 1u);
      if (any && zb + r < nz) atomicOr(hw + (r >> 5), 1u << (r & 31));
    }
    __syncthreads();
    if (tid < FB / 32 && hw[tid]) atomicOr(hit_words + (zb >> 5) + tid, hw[tid]);
    return;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int cj = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long zi = zb + ty * 4 + i;
      if (zi < nz && ((okmask >> (i * 4 + j)) & 1u)) ++cj;
    }
    cnt[ty][tx * 4 + j] = cj;
  }
  __syncthreads();
  if (tid < FB) {
    int s = 0;
#pragma unroll
    for (int t = 0; t < 16; ++t) s += cnt[t][tid];
    const long long xi = xb + tid;
    if (xi < nx && s) atomicAdd(counts + (row_perm ? row_perm[xi] : xi), s);
  }
}


// =============================================================================================
// Fantasy mode, FP64 on the tensor cores (north_star "FP64 tensor-core mode"; sm_100a has no FP64 tcgen05 path, so this
// is DMMA, mma.sync.m8n8k4.f64, as in the posterior solve).  CTA = 128 candidates x 64 unsafe points, 8 warps of 32 x 32,
// K chunks of 16 through a 3-stage cp.async ring (row stride 20 doubles: conflict-free fragment loads), 2 CTAs per SM.
// Both operands are K-major rows (Vx[c][x][k], Vz[c][z][k]), which is exactly the row.col fragment layout.  Per
// constraint: acc = v_x . v_z, then the same FP64 epilogue as k_fantasy_f64 (identical operations and order, so the two
// kernels agree bit for bit up to the summation order of the dot product); the decision bits are ANDed over the
// constraints in registers and counted per candidate with two shuffles + one atomicAdd.  Work items come from the same
// exact-pruning list as the tcgen05 kernels (fantasy_build_items).
// =============================================================================================
#define FD_BM 128
#define FD_BN 64
#define FD_BK 16
#define FD_LD 20
#define FD_STAGES 3
#define FD_STAGE_D ((FD_BM + FD_BN) * FD_LD)

struct DmmaArgs {
  long long nx, nz, nxp, nzp, n_items;
  int np, nxt, nzt, gx;
  const double *Vx, *Vz, *xn, *ax, *bx, *zn, *mz, *sz;
  int* counts;
  const int* row_perm;
  const long long* item_list;
  uint32_t* hit_words;          // GoOSE target: column OR over the candidates instead of counts
};

__device__ __forceinline__ void fd_cp16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void fd_dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

template <int D, bool TARGET, class KC>   // TARGET: GoOSE target epilogue (column OR into a.hit_words); KC: covariance function
__global__ void __launch_bounds__(256, 2)
k_fantasy_dmma(FantasyConsts fc, DmmaArgs a) {
  extern __shared__ __align__(16) double fsm[];
  const KC kc(fc.kernel);
  const int RC = D + 2 * fc.nc;                       // constants per row / column: xn[D] | a[nc] | b[nc]  (zn | m | s)
  double* rowc = fsm + FD_STAGES * FD_STAGE_D;        // [FD_BM][RC]
  double* colc = rowc + FD_BM * RC;                   // [FD_BN][RC]
  const long long item = a.item_list ? a.item_list[blockIdx.x] : (long long)blockIdx.x;
  const long long per_group = (long long)a.gx * a.nzt;
  const int xg = (int)(item / per_group), rr = (int)(item % per_group);
  const int zt = rr / a.gx, xt = xg * a.gx + rr % a.gx;
  if (xt >= a.nxt) return;
  const long long xb = (long long)xt * FD_BM, zb = (long long)zt * FD_BN;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int grp = lane >> 2, tig = lane & 3;
  const int wr = warp & 3, wp = warp >> 2;
  const int np = a.np, nc = fc.nc;
  for (int e = tid; e < FD_BM * RC; e += 256) {
    const int r = e / RC, k = e - r * RC;
    const long long xi = xb + r;
    double v = 0.0;
    if (xi < a.nx) v = k < D ? a.xn[(size_t)k * a.nx + xi] : (k < D + nc ? a.ax[(size_t)(k - D) * a.nx + xi] : a.bx[(size_t)(k - D - nc) * a.nx + xi]);
    rowc[e] = v;
  }
  for (int e = tid; e < FD_BN * RC; e += 256) {
    const int r = e / RC, k = e - r * RC;
    const long long zi = zb + r;
    double v = 0.0;
    if (zi < a.nz) v = k < D ? a.zn[(size_t)k * a.nz + zi] : (k < D + nc ? a.mz[(size_t)(k - D) * a.nz + zi] : a.sz[(size_t)(k - D - nc) * a.nz + zi]);
    colc[e] = v;
  }
  uint32_t okbits = 0xffffffffu;                      // bit (i*4 + j)*2 + e
  const int nk = np / FD_BK;
  for (int c = 0; c < nc; ++c) {
    const double* Xg = a.Vx + ((size_t)c * a.nxp + xb) * np;
    const double* Zg = a.Vz + ((size_t)c * a.nzp + zb) * np;
    auto load_chunk = [&](int stage, int k0) {
      double* Xs = fsm + stage * FD_STAGE_D;
      double* Zs = Xs + FD_BM * FD_LD;
#pragma unroll
      for (int q = 0; q < 4; ++q) {                   // 128 rows x 16 doubles = 1024 x 16 B
        const int e = tid + 256 * q, r = e >> 3, c2 = (e & 7) * 2;
        fd_cp16(Xs + r * FD_LD + c2, Xg + (size_t)r * np + k0 + c2);
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {                   // 64 rows x 16 doubles = 512 x 16 B
        const int e = tid + 256 * q, r = e >> 3, c2 = (e & 7) * 2;
        fd_cp16(Zs + r * FD_LD + c2, Zg + (size_t)r * np + k0 + c2);
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    __syncthreads();                                   // constants visible; stages free (previous constraint finished)
    load_chunk(0, 0);
    if (nk > 1) load_chunk(1, FD_BK);
    for (int kc = 0; kc < nk; ++kc) {
      if (kc + 2 < nk) {
        load_chunk((kc + 2) % FD_STAGES, (kc + 2) * FD_BK);
        asm volatile("cp.async.wait_group 2;" ::: "memory");
      } else if (kc + 1 < nk) {
        asm volatile("cp.async.wait_group 1;" ::: "memory");
      } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
      __syncthreads();
      const double* Xs = fsm + (kc % FD_STAGES) * FD_STAGE_D;
      const double* Zs = Xs + FD_BM * FD_LD;
#pragma unroll
      for (int k0 = 0; k0 < FD_BK; k0 += 4) {
        double av[4], bv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) av[i] = Xs[(wr * 32 + i * 8 + grp) * FD_LD + k0 + tig];
#pragma unroll
        for (int j = 0; j < 4; ++j) bv[j] = Zs[(wp * 32 + j * 8 + grp) * FD_LD + k0 + tig];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) fd_dmma(acc[i][j][0], acc[i][j][1], av[i], bv[j]);
      }
      __syncthreads();                                 // the stage is refilled two iterations later
    }
    // epilogue of constraint c: acc[i][j][e] = v_x . v_z for x row wr*32+i*8+grp, z column wp*32+j*8+2*tig+e
    const double sf2 = fc.sf2[c], beta = fc.beta;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const double* rx = rowc + (wr * 32 + i * 8 + grp) * RC;
      const double a_x = rx[D + c], b_x = rx[D + nc + c];
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const double* cz = colc + (wp * 32 + j * 8 + 2 * tig + e) * RC;
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < D; ++k) { const double df = cz[k] - rx[k]; s += df * df * fc.inv_ell[c][k]; }
          const double cc = kc.value(s, sf2) - acc[i][j][e];
          const double mu = cz[D + c] + cc * a_x;
          const double s2 = cz[D + nc + c] - cc * cc * b_x;
          if (!((mu - beta * sqrt(fmax(s2, 0.0))) >= 0.0)) okbits &= ~(1u << ((i * 4 + j) * 2 + e));
        }
    }
  }
  if (TARGET) {
    // GoOSE target: the warp's 32 z columns zb + wp*32 + (j*8 + 2*tig + e), OR over its valid x rows, one word per warp
    uint32_t w = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (xb + wr * 32 + i * 8 + grp >= a.nx) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int e = 0; e < 2; ++e)
          if (((okbits >> ((i * 4 + j) * 2 + e)) & 1u) && zb + wp * 32 + j * 8 + 2 * tig + e < a.nz) w |= 1u << (j * 8 + 2 * tig + e);
    }
    w = __reduce_or_sync(0xffffffffu, w);
    if (lane == 0 && w) atomicOr(a.hit_words + ((zb + wp * 32) >> 5), w);
    return;
  }
  // per candidate: newly-safe z of this tile = set bits of its row over valid columns, summed over the 4 lanes of a
  // quad (tig) here and over the two column warps by the atomics
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e)
        if (((okbits >> ((i * 4 + j) * 2 + e)) & 1u) && zb + wp * 32 + j * 8 + 2 * tig + e < a.nz) ++cnt;
    cnt += __shfl_xor_sync(0xffffffffu, cnt, 1);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, 2);
    const long long xi = xb + wr * 32 + i * 8 + grp;
    if (tig == 0 && cnt && xi < a.nx) atomicAdd(a.counts + (a.row_perm ? a.row_perm[xi] : xi), cnt);
  }
}

int fantasy_build_items(sbo_ctx* ctx, long long nx, long long nz, int tile_x, int tile_z, int gx, const double* key_x,
                        const double* key_z, const long long** item_list, long long* n_list);

struct FantasyPruneArgs { const double* key_x; const double* key_z; const int* row_perm; long long* items_run;
                          int refine; int2* amb_list; unsigned long long* amb_count; long long amb_cap; int* amb_rows;
                          uint32_t* hit_words; uint32_t* amb_words; };
int fantasy_tc_run(sbo_ctx* ctx, const FantasyConsts& fc, int split, long long nx, long long nz, long long nxp,
                   long long nzp, const float* Vx, const float* Vz, const double* aux_x, const double* aux_z, int* counts_c,
                   const FantasyPruneArgs* pr);


// =============================================================================================
// FP64 re-evaluation of the pairs the split-TF32 GEMM could not settle (fantasy_tc.cu epilogue_chunk_refine).
//   1. mark the distinct candidate slots / z columns of the ambiguous list, compact them, build slot -> rank maps
//   2. FP64 rows V = L^-1 K(X, .) for those points only (posterior kernels on explicit points)
//   3. one warp per ambiguous pair: FP64 dot products + the FP64 epilogue of k_fantasy_f64; safe pairs are added to the
//      candidate's count.  The GEMM counted only the pairs that are safe for EVERY covariance inside the error bound, so
//      the total equals the FP64 count (up to pairs within FP64 rounding of the threshold).
// =============================================================================================
__global__ void __launch_bounds__(256) k_amb_mark(long long n, const int2* __restrict__ list, uint32_t* __restrict__ xm, uint32_t* __restrict__ zm) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int2 e = list[t];
  atomicOr(xm + (e.x >> 5), 1u << (e.x & 31));
  atomicOr(zm + (e.y >> 5), 1u << (e.y & 31));
}
// rank[slot] = position in the compacted list; pts[r][d] = raw coordinates (xn * Xstd + Xmean)
__global__ void __launch_bounds__(256) k_amb_points(ModelSpec ms, long long m, long long ntot, const long long* __restrict__ ids,
                                                    const double* __restrict__ xn_soa, int* __restrict__ rank, double* __restrict__ pts) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= m) return;
  const long long id = ids[r];
  rank[id] = (int)r;
  for (int k = 0; k < ms.d; ++k) pts[(size_t)r * ms.d + k] = xn_soa[(size_t)k * ntot + id] * ms.Xstd[k] + ms.Xmean[k];
}
// ---------------------------------------------------------------------------------------------
// Cell-wise pass for lists whose points' FP64 rows do not fit the device at once (C5: ~1.6 M + 1.6 M rows of 49 KB per
// rank).  The compacted points are ranked, so a block is a contiguous rank range and cell = (outer block, inner block).
// The list is bucketed by cell (histogram, exclusive scan, scatter; the order inside a cell is arbitrary and no count
// depends on it); every outer block's rows are computed once, the inner blocks' rows once per outer block that pairs
// with them.  Every pair is evaluated by the same k_refine_pairs arithmetic on the same FP64 rows as in one cell.
// ---------------------------------------------------------------------------------------------
struct CellPlan {
  int bx, bz;              // block lengths in ranks (candidates, unsafe points)
  long long nbx, nbz;      // blocks per side
  bool z_outer;            // the z blocks form the outer loop (their rows are computed once)
};
__device__ __forceinline__ long long cell_of(const CellPlan& p, const int* __restrict__ rank_x, const int* __restrict__ rank_z, int2 e) {
  const long long cx = rank_x[e.x] / p.bx, cz = rank_z[e.y] / p.bz;
  return p.z_outer ? cz * p.nbx + cx : cx * p.nbz + cz;
}
__global__ void __launch_bounds__(256)
k_cell_hist(long long n, const int2* __restrict__ list, CellPlan p, const int* __restrict__ rank_x, const int* __restrict__ rank_z,
            int* __restrict__ hist) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) atomicAdd(hist + cell_of(p, rank_x, rank_z, list[t]), 1);
}
__global__ void __launch_bounds__(256)
k_cell_scatter(long long n, const int2* __restrict__ list, CellPlan p, const int* __restrict__ rank_x, const int* __restrict__ rank_z,
               int* __restrict__ cursor, int2* __restrict__ out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int2 e = list[t];
  out[atomicAdd(cursor + cell_of(p, rank_x, rank_z, e), 1)] = e;
}

// one warp per ambiguous pair of list[0..n_amb).  Vx / Vz hold the FP64 rows of the ranks [x0, x0 + mx) / [z0, z0 + mz_)
// (one cell: all ranks, offsets 0)
template <int D, bool TARGET, class KC>   // TARGET: GoOSE target (safe pairs set their z's bit in hit_words); KC: covariance function
__global__ void __launch_bounds__(256)
k_refine_pairs(FantasyConsts fc, long long n_amb, const int2* __restrict__ list, long long nx, long long nz, long long mx, long long mz_,
               long long x0, long long z0, const int* __restrict__ rank_x, const int* __restrict__ rank_z,
               const double* __restrict__ Vx, const double* __restrict__ Vz,
               const double* __restrict__ xn, const double* __restrict__ ax, const double* __restrict__ bx,
               const double* __restrict__ zn, const double* __restrict__ mz, const double* __restrict__ sz,
               int* __restrict__ counts, const int* __restrict__ row_perm, unsigned long long* __restrict__ n_safe,
               uint32_t* __restrict__ hit_words) {
  const long long w = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (w >= n_amb) return;
  const KC kc(fc.kernel);
  const int lane = threadIdx.x & 31;
  const int2 e = list[w];
  const long long xi = e.x, zi = e.y;
  const uint32_t zbit = 1u << (zi & 31);
  // GoOSE target: a pair can only re-confirm a z another pair of this pass already added (warp-uniform skip)
  if (TARGET && (*(volatile const uint32_t*)(hit_words + (zi >> 5)) & zbit)) return;
  const long long rx = rank_x[xi] - x0, rz = rank_z[zi] - z0;
  bool ok = true;
  for (int c = 0; c < fc.nc && ok; ++c) {
    const double* vx = Vx + ((size_t)c * mx + rx) * fc.npad;
    const double* vz = Vz + ((size_t)c * mz_ + rz) * fc.npad;
    double acc = 0.0;
    for (int k = lane; k < fc.npad; k += 32) acc = fma(vx[k], vz[k], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < D; ++k) { const double df = zn[(size_t)k * nz + zi] - xn[(size_t)k * nx + xi]; s += df * df * fc.inv_ell[c][k]; }
    const double cc = kc.value(s, fc.sf2[c]) - acc;
    const double mu = mz[(size_t)c * nz + zi] + cc * ax[(size_t)c * nx + xi];
    const double s2 = sz[(size_t)c * nz + zi] - cc * cc * bx[(size_t)c * nx + xi];
    ok = (mu - fc.beta * sqrt(fmax(s2, 0.0))) >= 0.0;
  }
  if (ok && lane == 0) {
    if (TARGET) {   // n_safe counts points: exactly one atomicOr sees the bit of a newly added z clear
      if (!(atomicOr(hit_words + (zi >> 5), zbit) & zbit)) atomicAdd(n_safe, 1ULL);
    } else {
      atomicAdd(counts + (row_perm ? row_perm[xi] : xi), 1);
      atomicAdd(n_safe, 1ULL);
    }
  }
}

static int launch_refine(sbo_ctx* ctx, const FantasyConsts& fc, long long n, const int2* list, long long nx, long long nz,
                         long long mx, long long mz_, long long x0, long long z0, const double* Vx, const double* Vz,
                         int* counts, const int* row_perm, uint32_t* hit_words) {
  const int d = fc.d, nc = fc.nc;
  const double* xn = (const double*)ctx->aux_x.p; const double* ax = xn + (size_t)d * nx; const double* bx = ax + (size_t)nc * nx;
  const double* zn = (const double*)ctx->aux_z.p; const double* mz = zn + (size_t)d * nz; const double* sz = mz + (size_t)nc * nz;
  unsigned long long* nsafe = (unsigned long long*)ctx->amb_ctr.p + 1;
  with_int<1, SBO_MAX_D>(d, [&](auto D) { with_flag(hit_words != nullptr, [&](auto T) { with_kernel(fc.kernel, [&](auto kc) {
    k_refine_pairs<D, T, decltype(kc)><<<(unsigned)cdiv(n, 8), 256, 0, ctx->stream>>>(fc, n, list, nx, nz, mx, mz_, x0, z0,
        (const int*)ctx->amb_rx.p, (const int*)ctx->amb_rz.p, Vx, Vz, xn, ax, bx, zn, mz, sz, counts, row_perm, nsafe, hit_words);
  }); }); });
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

#define REFINE_RESERVE ((size_t)1 << 30)        // automatic budget: device memory left to everything else
#define REFINE_MAX_CELLS (1LL << 22)

// FP64 rows + posterior scratch + buckets of a multi-cell pass with blocks (bx, bz)
static size_t cell_pass_bytes(const sbo_ctx* ctx, long long n_amb, size_t row_b, long long bx, long long bz, long long cells) {
  size_t mv, kb;
  posterior_vrows_scratch(ctx, bx > bz ? bx : bz, &mv, &kb);
  return (size_t)(bx + bz) * row_b + 2 * mv + kb + sizeof(int2) * (size_t)n_amb + sizeof(int) * 2 * (size_t)cells;
}

// the largest blocks whose pass fits `budget`: the inner side gets a quarter of the rows (all of its ranks if fewer), the
// outer side the rest; of the two orientations the one that computes fewer rows (outer once, inner once per outer block)
static bool plan_cells(const sbo_ctx* ctx, long long mx, long long mz, long long n_amb, size_t row_b, size_t budget, CellPlan* best) {
  const size_t fixed = sizeof(int2) * (size_t)n_amb;
  if (budget <= fixed + 2 * row_b) return false;
  for (long long R = (long long)((budget - fixed) / row_b); R >= 2; R -= R / 8 > 1 ? R / 8 : 1) {
    long long best_rows = -1;
    for (int zo = 0; zo < 2; ++zo) {
      const long long mo = zo ? mz : mx, mi = zo ? mx : mz;
      long long bi = mi < R / 4 ? mi : (R / 4 > 1 ? R / 4 : 1);
      const long long bo = mo < R - bi ? mo : R - bi;
      bi = mi < R - bo ? mi : R - bo;
      const long long no = cdiv(mo, bo), ni = cdiv(mi, bi);
      if (bo > 2000000000LL || bi > 2000000000LL || no * ni > REFINE_MAX_CELLS) continue;
      const long long rows = mo + mi * no;
      CellPlan p{(int)(zo ? bi : bo), (int)(zo ? bo : bi), zo ? ni : no, zo ? no : ni, zo == 1};
      if (cell_pass_bytes(ctx, n_amb, row_b, p.bx, p.bz, no * ni) > budget) continue;
      if (best_rows < 0 || rows < best_rows) { best_rows = rows; *best = p; }
    }
    if (best_rows >= 0) return true;
  }
  return false;
}

// GoOSE target: the listed pairs whose z is not yet in the target set (the order of the kept pairs is arbitrary)
__global__ void __launch_bounds__(256) k_amb_filter(long long n, const int2* __restrict__ list, const uint32_t* __restrict__ hit_words,
                                                    int2* __restrict__ out, unsigned long long* __restrict__ n_out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int2 e = list[t];
  if (!((hit_words[e.y >> 5] >> (e.y & 31)) & 1u)) out[atomicAdd(n_out, 1ULL)] = e;
}

// counts != null: SafeOpt expander (safe pairs are added to the candidates' counts).  hit_words != null: GoOSE target (safe
// pairs set their z's bit; the list is first cut to the pairs whose z no settled pair reached, and n_refined_safe counts the
// unsafe points the pass adds to the target set)
static int refine_ambiguous(sbo_ctx* ctx, const FantasyConsts& fc, long long nx, long long nz, int* counts, const int* row_perm,
                            uint32_t* hit_words) {
  PairStage& ps = ctx->ps;
  const ModelSpec& ms = ctx->ms;
  const int d = fc.d, nc = fc.nc;
  unsigned long long h[2] = {0, 0};
  SBO_CUDA(cudaMemcpyAsync(h, ctx->amb_ctr.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  long long n_amb = (long long)h[0];
  const long long cap = (long long)(ctx->amb_list.cap / sizeof(int2));
  ps.n_ambiguous = n_amb; ps.n_refined_safe = 0;
  if (n_amb > cap)
    return sbo_fail(ctx, SBO_ERR_NOMEM, "split-TF32 refinement: " + std::to_string(n_amb) + " ambiguous pairs exceed the list capacity " +
                                            std::to_string(cap) + " (use precision fp64, or option fantasy_refine = 0)");
  if (n_amb == 0) return SBO_OK;
  const int2* list = (const int2*)ctx->amb_list.p;
  if (hit_words) {
    SBO_TRY(sbo_ensure(ctx, ctx->amb_tgt, sizeof(int2) * (size_t)n_amb));
    SBO_CUDA(cudaMemsetAsync(ctx->amb_ctr.p, 0, sizeof(unsigned long long), ctx->stream));
    k_amb_filter<<<(unsigned)cdiv(n_amb, 256), 256, 0, ctx->stream>>>(n_amb, list, hit_words, (int2*)ctx->amb_tgt.p, (unsigned long long*)ctx->amb_ctr.p);
    SBO_LAUNCH_CHECK();
    SBO_CUDA(cudaMemcpyAsync(h, ctx->amb_ctr.p, sizeof(h[0]), cudaMemcpyDeviceToHost, ctx->stream));
    SBO_CUDA(cudaStreamSynchronize(ctx->stream));
    n_amb = (long long)h[0];
    list = (const int2*)ctx->amb_tgt.p;
    if (n_amb == 0) return SBO_OK;
  }
  const long long wx = cdiv(nx, 32), wz = cdiv(nz, 32);
  SBO_TRY(sbo_ensure(ctx, ctx->amb_mask, sizeof(uint32_t) * (size_t)(wx + wz)));
  SBO_CUDA(cudaMemsetAsync(ctx->amb_mask.p, 0, sizeof(uint32_t) * (size_t)(wx + wz), ctx->stream));
  uint32_t* xm = (uint32_t*)ctx->amb_mask.p; uint32_t* zm = xm + wx;
  k_amb_mark<<<(unsigned)cdiv(n_amb, 256), 256, 0, ctx->stream>>>(n_amb, list, xm, zm);
  SBO_LAUNCH_CHECK();
  long long mx = 0, mzd = 0;
  SBO_TRY(compact_mask(ctx, xm, nx, ctx->amb_xd, &mx));
  SBO_TRY(compact_mask(ctx, zm, nz, ctx->amb_zd, &mzd));
  SBO_TRY(sbo_ensure(ctx, ctx->amb_rx, sizeof(int) * (size_t)nx));
  SBO_TRY(sbo_ensure(ctx, ctx->amb_rz, sizeof(int) * (size_t)nz));
  SBO_TRY(sbo_ensure(ctx, ctx->amb_pts, sizeof(double) * (size_t)(mx + mzd) * d));
  const double* xn = (const double*)ctx->aux_x.p;
  const double* zn = (const double*)ctx->aux_z.p;
  double* ptx = (double*)ctx->amb_pts.p; double* ptz = ptx + (size_t)mx * d;
  k_amb_points<<<(unsigned)cdiv(mx, 256), 256, 0, ctx->stream>>>(ms, mx, nx, (const long long*)ctx->amb_xd.p, xn, (int*)ctx->amb_rx.p, ptx);
  SBO_LAUNCH_CHECK();
  k_amb_points<<<(unsigned)cdiv(mzd, 256), 256, 0, ctx->stream>>>(ms, mzd, nz, (const long long*)ctx->amb_zd.p, zn, (int*)ctx->amb_rz.p, ptz);
  SBO_LAUNCH_CHECK();

  // memory budget of the pass: option fantasy_refine_mb, or what is free now plus the buffers the pass (re)uses, less a reserve
  const size_t row_b = sizeof(double) * (size_t)nc * ms.npad;          // FP64 rows of one point, all constraints
  size_t free_b = 0, total_b = 0;
  SBO_CUDA(cudaMemGetInfo(&free_b, &total_b));
  size_t avail = free_b;
  for (const DevBuf* b : {&ctx->amb_vx, &ctx->amb_vz, &ctx->pp_m, &ctx->pp_v, &ctx->pp_k, &ctx->amb_cell, &ctx->amb_hist}) avail += b->cap;
  size_t budget = avail > REFINE_RESERVE ? avail - REFINE_RESERVE : 0;
  if (ctx->opt_fantasy_refine_mb > 0 && (size_t)ctx->opt_fantasy_refine_mb << 20 < budget) budget = (size_t)ctx->opt_fantasy_refine_mb << 20;
  size_t mv1, kb1;
  posterior_vrows_scratch(ctx, mx > mzd ? mx : mzd, &mv1, &kb1);
  const size_t one_cell = (size_t)(mx + mzd) * row_b + 2 * mv1 + kb1;

  const bool multi = one_cell > budget;
  if (!multi) {
    // one cell: every row at once (the buffers keep sbo_ensure's head-room when the budget has it)
    const bool room = one_cell + one_cell / 8 <= budget;
    SBO_TRY((room ? sbo_ensure : sbo_ensure_exact)(ctx, ctx->amb_vx, sizeof(double) * (size_t)nc * mx * ms.npad));
    SBO_TRY((room ? sbo_ensure : sbo_ensure_exact)(ctx, ctx->amb_vz, sizeof(double) * (size_t)nc * mzd * ms.npad));
    if (!room) {
      SBO_TRY(sbo_ensure_exact(ctx, ctx->pp_m, mv1)); SBO_TRY(sbo_ensure_exact(ctx, ctx->pp_v, mv1)); SBO_TRY(sbo_ensure_exact(ctx, ctx->pp_k, kb1));
    }
    SBO_TRY(posterior_vrows_dev(ctx, mx, ptx, (double*)ctx->amb_vx.p));
    SBO_TRY(posterior_vrows_dev(ctx, mzd, ptz, (double*)ctx->amb_vz.p));
    SBO_TRY(launch_refine(ctx, fc, n_amb, list, nx, nz, mx, mzd, 0, 0, (const double*)ctx->amb_vx.p, (const double*)ctx->amb_vz.p, counts, row_perm, hit_words));
    ctx->refine_cells = 1; ctx->refine_rows = mx + mzd;
  } else {
    CellPlan p{};
    if (!plan_cells(ctx, mx, mzd, n_amb, row_b, budget, &p))
      return sbo_fail(ctx, SBO_ERR_NOMEM, "split-TF32 refinement: " + std::to_string(budget >> 20) + " MB cannot hold the FP64 rows of one candidate "
                                              "and one unsafe point with their scratch (" + std::to_string(n_amb) + " ambiguous pairs); raise option "
                                              "fantasy_refine_mb (0 = the free device memory) or use fantasy_refine = 3");
    const long long ncell = p.nbx * p.nbz;
    // the budget was planned for exactly these buffers: drop what the context holds and allocate them without head-room
    for (DevBuf* b : {&ctx->amb_vx, &ctx->amb_vz, &ctx->pp_m, &ctx->pp_v, &ctx->pp_k, &ctx->amb_cell, &ctx->amb_hist}) sbo_free(ctx, *b);
    size_t mv, kb;
    posterior_vrows_scratch(ctx, p.bx > p.bz ? p.bx : p.bz, &mv, &kb);
    SBO_TRY(sbo_ensure_exact(ctx, ctx->amb_vx, row_b * (size_t)p.bx));
    SBO_TRY(sbo_ensure_exact(ctx, ctx->amb_vz, row_b * (size_t)p.bz));
    SBO_TRY(sbo_ensure_exact(ctx, ctx->pp_m, mv)); SBO_TRY(sbo_ensure_exact(ctx, ctx->pp_v, mv)); SBO_TRY(sbo_ensure_exact(ctx, ctx->pp_k, kb));
    SBO_TRY(sbo_ensure_exact(ctx, ctx->amb_cell, sizeof(int2) * (size_t)n_amb));
    SBO_TRY(sbo_ensure_exact(ctx, ctx->amb_hist, sizeof(int) * 2 * (size_t)ncell));
    // bucket the list by cell.  The host needs every cell's length to launch it, so the exclusive scan runs there
    int* hist = (int*)ctx->amb_hist.p; int* cursor = hist + ncell;
    int2* sorted = (int2*)ctx->amb_cell.p;
    const int* rkx = (const int*)ctx->amb_rx.p; const int* rkz = (const int*)ctx->amb_rz.p;
    SBO_CUDA(cudaMemsetAsync(hist, 0, sizeof(int) * (size_t)ncell, ctx->stream));
    k_cell_hist<<<(unsigned)cdiv(n_amb, 256), 256, 0, ctx->stream>>>(n_amb, list, p, rkx, rkz, hist);
    SBO_LAUNCH_CHECK();
    std::vector<int> cnt((size_t)ncell), off((size_t)ncell);
    SBO_CUDA(cudaMemcpyAsync(cnt.data(), hist, sizeof(int) * (size_t)ncell, cudaMemcpyDeviceToHost, ctx->stream));
    SBO_CUDA(cudaStreamSynchronize(ctx->stream));
    long long run = 0;
    for (long long c = 0; c < ncell; ++c) { off[c] = (int)run; run += cnt[c]; }
    SBO_CUDA(cudaMemcpyAsync(cursor, off.data(), sizeof(int) * (size_t)ncell, cudaMemcpyHostToDevice, ctx->stream));
    k_cell_scatter<<<(unsigned)cdiv(n_amb, 256), 256, 0, ctx->stream>>>(n_amb, list, p, rkx, rkz, cursor, sorted);
    SBO_LAUNCH_CHECK();
    // outer blocks: rows once; inner blocks: rows for every outer block they have pairs with (empty cells are skipped)
    const long long no = p.z_outer ? p.nbz : p.nbx, ni = p.z_outer ? p.nbx : p.nbz;
    long long cells = 0, rows = 0;
    for (long long o = 0; o < no; ++o) {
      long long in_block = 0;
      for (long long i = 0; i < ni; ++i) in_block += cnt[(size_t)(o * ni + i)];
      if (in_block == 0) continue;
      const long long b_o = p.z_outer ? p.bz : p.bx, m_o = p.z_outer ? mzd : mx;
      const long long r0 = o * b_o, len_o = (m_o - r0) < b_o ? (m_o - r0) : b_o;
      SBO_TRY(posterior_vrows_dev(ctx, len_o, (p.z_outer ? ptz : ptx) + (size_t)r0 * d, (double*)(p.z_outer ? ctx->amb_vz.p : ctx->amb_vx.p)));
      rows += len_o;
      for (long long i = 0; i < ni; ++i) {
        const long long c = o * ni + i;
        if (cnt[(size_t)c] == 0) continue;
        const long long b_i = p.z_outer ? p.bx : p.bz, m_i = p.z_outer ? mx : mzd;
        const long long q0 = i * b_i, len_i = (m_i - q0) < b_i ? (m_i - q0) : b_i;
        SBO_TRY(posterior_vrows_dev(ctx, len_i, (p.z_outer ? ptx : ptz) + (size_t)q0 * d, (double*)(p.z_outer ? ctx->amb_vx.p : ctx->amb_vz.p)));
        rows += len_i;
        const long long x0 = p.z_outer ? q0 : r0, lx = p.z_outer ? len_i : len_o;
        const long long z0 = p.z_outer ? r0 : q0, lz = p.z_outer ? len_o : len_i;
        SBO_TRY(launch_refine(ctx, fc, cnt[(size_t)c], sorted + off[(size_t)c], nx, nz, lx, lz, x0, z0,
                              (const double*)ctx->amb_vx.p, (const double*)ctx->amb_vz.p, counts, row_perm, hit_words));
        ++cells;
      }
    }
    ctx->refine_cells = cells; ctx->refine_rows = rows;
  }
  SBO_CUDA(cudaMemcpyAsync(h, ctx->amb_ctr.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  ps.n_refined_safe = (long long)h[1];
  if (multi)      // up to tens of GB (C5): the next step's posterior needs them
    for (DevBuf* b : {&ctx->amb_vx, &ctx->amb_vz, &ctx->amb_cell}) sbo_free(ctx, *b);
  return SBO_OK;
}

// =============================================================================================
// staged host driver
// =============================================================================================
static int vrow_elems(const sbo_ctx* ctx) {   // V elements per candidate per constraint
  return ctx->ps.precision == SBO_PREC_TF32X3 ? 2 * ctx->ms.npad : ctx->ms.npad;
}
static size_t v_elem_size(const sbo_ctx* ctx) { return ctx->ps.precision == SBO_PREC_FP64 ? sizeof(double) : sizeof(float); }

int pairs_prepare(sbo_ctx* ctx, int mode, int precision, double beta, const double* L, sbo_pairs_info* info) {
  SBO_REQUIRE(ctx->have_sets, "pair kernels need the sets (call sbo_sets / sbo_sets_pass1)");
  SBO_REQUIRE(mode == SBO_MODE_LIPSCHITZ || mode == SBO_MODE_FANTASY, "bad expander mode");
  const ModelSpec& ms = ctx->ms;
  const GridSpec& gs = ctx->gs;
  const int nc = ms.G - 1, d = gs.d;
  const long long count = gs.count;
  PairStage& ps = ctx->ps;
  stage_changed(ctx, Change::PAIRS);
  ctx->refine_cells = ctx->refine_rows = 0;
  ps.mode = mode; ps.precision = precision; ps.beta = beta;
  ps.row_doubles = 2 * d + 3 * nc + 1;
  if (mode == SBO_MODE_LIPSCHITZ) {
    SBO_REQUIRE(L != nullptr || nc == 0, "Lipschitz constants required");
    for (int c = 0; c < nc; ++c) ps.L[c] = L[c + 1];
  } else {
    SBO_REQUIRE(nc >= 1, "fantasy expander needs at least one constraint GP");
    SBO_REQUIRE(precision == SBO_PREC_FP64 || precision == SBO_PREC_TF32 || precision == SBO_PREC_TF32X3, "bad precision");
    SBO_REQUIRE(ctx->keep_v == keep_v_of(precision),
                "fantasy expander: run sbo_posterior with keep_v = 1 (FP64), 2 (TF32) or 3 (TF32x3) first");
  }
  ev_reset(ctx, 4); ev_reset(ctx, 6); ev_reset(ctx, 7);
  ev_begin(ctx, 6);
  long long nx = 0, nz = 0;
  ps.nz_full = 0;
  if (nc > 0) {
    SBO_TRY(compact_mask(ctx, (const uint32_t*)ctx->m_safe.p, count, ctx->xs_idx, &nx));
    SBO_TRY(compact_mask(ctx, (const uint32_t*)ctx->m_unsafe.p, count, ctx->zs_idx, &nz));
    ps.nz_full = nz;
    if (mode == SBO_MODE_FANTASY && ctx->opt_fantasy_prune && nz > 0) {
      // order the unsafe points by key_z = max_c rho_zc and drop those no candidate can reach (key_z > 1)
      SBO_TRY(sbo_ensure(ctx, ctx->key_z, sizeof(double) * (size_t)nz * 2));
      double* kz = (double*)ctx->key_z.p;
      k_key_z<<<(unsigned)cdiv(nz, 256), 256, 0, ctx->stream>>>(ms.G, count, beta, ms, (const long long*)ctx->zs_idx.p, nz,
                                                               (const double*)ctx->mean.p, (const double*)ctx->var.p, kz + nz);
      SBO_LAUNCH_CHECK();
      long long keep = nz;
      SBO_TRY(sort_by_key(ctx, nz, kz + nz, ctx->perm_z, &keep));
      SBO_TRY(sbo_ensure(ctx, ctx->scan_b, sizeof(long long) * (size_t)nz));
      k_permute_idx<<<(unsigned)cdiv(nz, 256), 256, 0, ctx->stream>>>(nz, (const int*)ctx->perm_z.p, (const long long*)ctx->zs_idx.p, (long long*)ctx->scan_b.p);
      SBO_LAUNCH_CHECK();
      k_permute_key<<<(unsigned)cdiv(nz, 256), 256, 0, ctx->stream>>>(nz, (const int*)ctx->perm_z.p, kz + nz, kz);
      SBO_LAUNCH_CHECK();
      std::swap(ctx->zs_idx, ctx->scan_b);          // zs_idx is now in key order; kz[0..nz) the sorted keys
      nz = keep;
      ps.sorted = true;
    }
  }
  ps.nx_local = nx; ps.nz_local = nz;
  if (nz > 0) {   // local Z-side payload
    const long long* zi = (const long long*)ctx->zs_idx.p;
    if (mode == SBO_MODE_LIPSCHITZ) {
      SBO_TRY(sbo_ensure(ctx, ctx->zs_pay, sizeof(double) * (size_t)nz * d));
      k_gather_coords<<<(unsigned)cdiv(nz, 256), 256, 0, ctx->stream>>>(gs, zi, nz, (double*)ctx->zs_pay.p);
      SBO_LAUNCH_CHECK();
    } else {
      const int rowlen = vrow_elems(ctx);
      const long long nzp = cdiv(nz, 256) * 256;
      SBO_TRY(sbo_ensure(ctx, ctx->vz, v_elem_size(ctx) * (size_t)nc * nzp * rowlen));
      SBO_TRY(sbo_ensure(ctx, ctx->aux_z, sizeof(double) * (size_t)nz * (d + 2 * nc)));
      if (precision == SBO_PREC_FP64)
        k_gather_rows<double><<<dim3((unsigned)cdiv(nzp, 8), nc), 256, 0, ctx->stream>>>(nc, rowlen, nz, nzp, count, zi, (const double*)ctx->vall.p, (double*)ctx->vz.p);
      else
        k_gather_rows<float><<<dim3((unsigned)cdiv(nzp, 8), nc), 256, 0, ctx->stream>>>(nc, rowlen, nz, nzp, count, zi, (const float*)ctx->vall.p, (float*)ctx->vz.p);
      SBO_LAUNCH_CHECK();
      double* zn = (double*)ctx->aux_z.p; double* mz = zn + (size_t)d * nz; double* sz = mz + (size_t)nc * nz;
      k_fantasy_aux_z<<<(unsigned)cdiv(nz, 256), 256, 0, ctx->stream>>>(gs, ms, zi, nz, (const double*)ctx->mean.p, (const double*)ctx->var.p, zn, mz, sz);
      SBO_LAUNCH_CHECK();
    }
  }
  ev_end(ctx);
  stage_changed(ctx, Change::PAIRS_PREPARED);
  if (info) {
    info->n_x_local = nx; info->n_z_local = ps.nz_full; info->row_doubles = ps.row_doubles;
    info->vrow_bytes = (mode == SBO_MODE_FANTASY) ? (int64_t)(v_elem_size(ctx) * (size_t)nc * vrow_elems(ctx)) : 0;
  }
  return SBO_OK;
}

int pairs_export(sbo_ctx* ctx, void* rows_dev, void* vrows_dev) {
  PairStage& ps = ctx->ps;
  SBO_REQUIRE(ps.exportable, "sbo_pairs_export: call sbo_pairs_prepare first");
  const long long nx = ps.nx_local;
  if (nx == 0) return SBO_OK;
  SBO_REQUIRE(rows_dev != nullptr, "null export buffer");
  const ModelSpec& ms = ctx->ms;
  const int nc = ms.G - 1;
  const long long* xi = (const long long*)ctx->xs_idx.p;
  ev_begin(ctx, 6);
  k_export_rows<<<(unsigned)cdiv(nx, 256), 256, 0, ctx->stream>>>(ctx->gs, ms, ps.beta, xi, nx, (const double*)ctx->mean.p,
                                                                  (const double*)ctx->var.p, (double*)rows_dev);
  SBO_LAUNCH_CHECK();
  if (ps.mode == SBO_MODE_FANTASY) {
    SBO_REQUIRE(vrows_dev != nullptr, "null V export buffer");
    const int rowlen = vrow_elems(ctx);
    if (ps.precision == SBO_PREC_FP64)
      k_export_v<double><<<dim3((unsigned)cdiv(nx, 8), nc), 256, 0, ctx->stream>>>(nc, rowlen, nx, ctx->gs.count, xi, (const double*)ctx->vall.p, (double*)vrows_dev);
    else
      k_export_v<float><<<dim3((unsigned)cdiv(nx, 8), nc), 256, 0, ctx->stream>>>(nc, rowlen, nx, ctx->gs.count, xi, (const float*)ctx->vall.p, (float*)vrows_dev);
    SBO_LAUNCH_CHECK();
  }
  ev_end(ctx);
  return SBO_OK;
}

int pairs_import(sbo_ctx* ctx, long long n_total, const void* rows_dev, const void* vrows_dev) {
  PairStage& ps = ctx->ps;
  SBO_REQUIRE(ps.prepared, "sbo_pairs_import: call sbo_pairs_prepare first");
  SBO_REQUIRE(n_total >= 0, "bad candidate count");
  ps.nx_total = n_total;
  stage_changed(ctx, Change::PAIRS_IMPORTED);
  if (n_total == 0) return SBO_OK;
  SBO_REQUIRE(rows_dev != nullptr, "null import buffer");
  const ModelSpec& ms = ctx->ms;
  const int nc = ms.G - 1, d = ctx->gs.d;
  PairConsts pc{};
  pc.nc = nc; pc.beta = ps.beta;
  for (int c = 0; c < nc; ++c) pc.L[c] = ps.L[c];
  // SoA payloads: xs_pay = coords[d] ucb[nc] thr[nc] ; aux_x = xn[d] ax[nc] bx[nc]
  SBO_TRY(sbo_ensure(ctx, ctx->xs_pay, sizeof(double) * (size_t)n_total * (d + 2 * nc)));
  SBO_TRY(sbo_ensure(ctx, ctx->aux_x, sizeof(double) * (size_t)n_total * (d + 2 * nc)));
  double* xc = (double*)ctx->xs_pay.p; double* ucb = xc + (size_t)d * n_total; double* thr = ucb + (size_t)nc * n_total;
  double* xn = (double*)ctx->aux_x.p; double* ax = xn + (size_t)d * n_total; double* bx = ax + (size_t)nc * n_total;
  ev_begin(ctx, 6);
  const int* xperm = nullptr;
  if (ps.sorted) {   // order ALL candidates by key_x = max_c q_xc (+ slack): see the pruning note above
    FantasyConsts fk{};
    fk.nc = nc;
    for (int c = 0; c < nc; ++c) fk.sn2[c] = ms.sn2[c + 1];
    SBO_TRY(sbo_ensure(ctx, ctx->key_x, sizeof(double) * (size_t)n_total * 2));
    double* kx = (double*)ctx->key_x.p;
    k_key_x<<<(unsigned)cdiv(n_total, 256), 256, 0, ctx->stream>>>(d, nc, n_total, fk, (const double*)rows_dev, kx + n_total);
    SBO_LAUNCH_CHECK();
    SBO_TRY(sort_by_key(ctx, n_total, kx + n_total, ctx->perm_x, nullptr));
    k_permute_key<<<(unsigned)cdiv(n_total, 256), 256, 0, ctx->stream>>>(n_total, (const int*)ctx->perm_x.p, kx + n_total, kx);
    SBO_LAUNCH_CHECK();
    xperm = (const int*)ctx->perm_x.p;
  } else if (ps.seg_n > 1 && n_total > 0) {
    // sharded Lipschitz run: restore grid order (spatially compact tiles for the bounding-box culling); the gathered rows
    // are rank-major and each rank's cyclic blocks are scattered over the grid
    SBO_REQUIRE(ps.seg_off[ps.seg_n] == n_total, "sbo_pairs_set_segments: the per-rank counts do not add up to n_total");
    SBO_TRY(sbo_ensure(ctx, ctx->perm_x, sizeof(int) * (size_t)n_total));
    SBO_TRY(sbo_ensure(ctx, ctx->sort_ws, sizeof(long long) * 64 + sizeof(int) * 2 * 4096 + 16));
    SBO_CUDA(cudaMemcpyAsync(ctx->sort_ws.p, ps.seg_off, sizeof(long long) * (ps.seg_n + 1), cudaMemcpyHostToDevice, ctx->stream));
    k_canon_perm<<<(unsigned)cdiv(n_total, 256), 256, 0, ctx->stream>>>(n_total, ps.seg_n, (const long long*)ctx->sort_ws.p,
                                                                          (const double*)rows_dev, ps.row_doubles, (int*)ctx->perm_x.p);
    SBO_LAUNCH_CHECK();
    xperm = (const int*)ctx->perm_x.p;
    ps.canon = true;
  }
  k_import_rows<<<(unsigned)cdiv(n_total, 256), 256, 0, ctx->stream>>>(d, nc, n_total, pc, xperm, (const double*)rows_dev, xc, ucb, thr, xn, ax, bx);
  SBO_LAUNCH_CHECK();
  if (ps.mode == SBO_MODE_FANTASY) {
    SBO_REQUIRE(vrows_dev != nullptr, "null V import buffer");
    const int rowlen = vrow_elems(ctx);
    const long long nxp = cdiv(n_total, 256) * 256;
    SBO_TRY(sbo_ensure(ctx, ctx->vx, v_elem_size(ctx) * (size_t)nc * nxp * rowlen));
    if (ps.precision == SBO_PREC_FP64)
      k_import_v<double><<<dim3((unsigned)cdiv(nxp, 8), nc), 256, 0, ctx->stream>>>(nc, rowlen, n_total, nxp, xperm, (const double*)vrows_dev, (double*)ctx->vx.p);
    else
      k_import_v<float><<<dim3((unsigned)cdiv(nxp, 8), nc), 256, 0, ctx->stream>>>(nc, rowlen, n_total, nxp, xperm, (const float*)vrows_dev, (float*)ctx->vx.p);
    SBO_LAUNCH_CHECK();
  }
  ev_end(ctx);
  return SBO_OK;
}

// sharded GoOSE target over the global unsafe list: flags of THIS rank's unsafe points, hits_local[c][t] = hits_global[c][pos]
// with pos = position of local point zs_idx[t] in the ascending global list (binary search)
__global__ void __launch_bounds__(256)
k_goose_localize(GridSpec gs, int nc, long long nz_local, const long long* __restrict__ zs_idx, const long long* __restrict__ gz_idx,
                 long long nz_global, const unsigned char* __restrict__ hg, unsigned char* __restrict__ hl) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nz_local) return;
  const long long g = shard_global(gs, zs_idx[t]);
  long long lo = 0, hi = nz_global;
  while (lo < hi) { const long long m = (lo + hi) >> 1; if (gz_idx[m] < g) lo = m + 1; else hi = m; }
  for (int c = 0; c < nc; ++c) hl[(size_t)c * nz_local + t] = (lo < nz_global && gz_idx[lo] == g) ? hg[(size_t)c * nz_global + lo] : 0;
}
int pairs_goose_localize(sbo_ctx* ctx, const void* hits_global, void* hits_local) {
  PairStage& ps = ctx->ps;
  SBO_REQUIRE(ps.prepared && ps.nz_global >= 0, "pairs_goose_localize: no global unsafe set");
  const int nc = ctx->ms.G - 1;
  if (ps.nz_local == 0 || nc == 0) return SBO_OK;
  k_goose_localize<<<(unsigned)cdiv(ps.nz_local, 256), 256, 0, ctx->stream>>>(ctx->gs, nc, ps.nz_local, (const long long*)ctx->zs_idx.p,
                                                                               (const long long*)ctx->gz_idx.p, ps.nz_global,
                                                                               (const unsigned char*)hits_global, (unsigned char*)hits_local);
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

int pairs_set_segments(sbo_ctx* ctx, int nranks, int rank, const int64_t* n_per_rank) {
  PairStage& ps = ctx->ps;
  SBO_REQUIRE(ps.prepared, "sbo_pairs_set_segments: call sbo_pairs_prepare first");
  SBO_REQUIRE(nranks >= 1 && nranks <= 64 && rank >= 0 && rank < nranks && n_per_rank, "bad segments");
  ps.seg_n = nranks; ps.seg_rank = rank;
  ps.seg_off[0] = 0;
  for (int r = 0; r < nranks; ++r) {
    SBO_REQUIRE(n_per_rank[r] >= 0, "negative candidate count");
    ps.seg_off[r + 1] = ps.seg_off[r] + n_per_rank[r];
  }
  return SBO_OK;
}

// gathered_words_dev: the ranks' LOCAL unsafe masks, words_per_rank words each (zero padded), rank-major
int pairs_set_global_unsafe(sbo_ctx* ctx, const void* gathered_words_dev, long long words_per_rank, int nranks) {
  PairStage& ps = ctx->ps;
  SBO_REQUIRE(ps.prepared && ps.mode == SBO_MODE_LIPSCHITZ, "sbo_pairs_set_global_unsafe_dev: prepare the Lipschitz pair stage first");
  const GridSpec& gs = ctx->gs;
  SBO_REQUIRE(nranks >= 1 && gathered_words_dev && words_per_rank >= 1, "bad gathered mask");
  SBO_REQUIRE(nranks == 1 || (gs.cyc_n == nranks && gs.cyc_blk % 32 == 0), "the grid must be sharded with sbo_set_shard_cyclic over the same ranks");
  const long long nwg = cdiv(gs.N, 32);
  SBO_TRY(sbo_ensure(ctx, ctx->gz_mask, sizeof(uint32_t) * (size_t)nwg));
  ev_begin(ctx, 6);
  if (nranks == 1) {
    SBO_CUDA(cudaMemcpyAsync(ctx->gz_mask.p, gathered_words_dev, sizeof(uint32_t) * (size_t)(nwg < words_per_rank ? nwg : words_per_rank),
                             cudaMemcpyDeviceToDevice, ctx->stream));
  } else {
    k_assemble_global_mask<<<(unsigned)cdiv(nwg, 256), 256, 0, ctx->stream>>>(nwg, gs.cyc_blk, nranks, (const uint32_t*)gathered_words_dev,
                                                                               words_per_rank, (uint32_t*)ctx->gz_mask.p);
    SBO_LAUNCH_CHECK();
  }
  long long nzg = 0;
  SBO_TRY(compact_mask(ctx, (const uint32_t*)ctx->gz_mask.p, gs.N, ctx->gz_idx, &nzg));
  if (nzg > 0) {
    SBO_TRY(sbo_ensure(ctx, ctx->gz_pay, sizeof(double) * (size_t)nzg * gs.d));
    k_gather_coords_global<<<(unsigned)cdiv(nzg, 256), 256, 0, ctx->stream>>>(gs, (const long long*)ctx->gz_idx.p, nzg, (double*)ctx->gz_pay.p);
    SBO_LAUNCH_CHECK();
  }
  ev_end(ctx);
  ps.nz_global = nzg;
  return SBO_OK;
}

// result_dev: expander/lipschitz uint8[nc*n_total]; expander/fantasy int32[n_total]; goose/lipschitz uint8[nc*nz_local];
// goose/fantasy uint32[ceil(nz_local/32)] hit words over the prepared (key-sorted) z slots
int pairs_run(sbo_ctx* ctx, int goose, void* result_dev) {
  PairStage& ps = ctx->ps;
  SBO_REQUIRE(ps.prepared && ps.imported, "sbo_pairs_run: prepare and import first");
  const ModelSpec& ms = ctx->ms;
  const int nc = ms.G - 1, d = ctx->gs.d;
  const long long nx = ps.nx_total, nz = ps.nz_local;
  ps.pairs_evaluated = 0;
  ps.counted = false;
  ps.bounds = false;
  if (nc == 0) return SBO_OK;
  const size_t res_bytes = (ps.mode == SBO_MODE_FANTASY) ? (goose ? sizeof(uint32_t) * (size_t)cdiv(nz, 32) : sizeof(int) * (size_t)nx)
                                                         : (size_t)nc * (goose ? (ps.nz_global >= 0 ? ps.nz_global : nz) : nx);
  if (res_bytes) {
    SBO_REQUIRE(result_dev != nullptr, "null result buffer");
    SBO_CUDA(cudaMemsetAsync(result_dev, 0, res_bytes, ctx->stream));
  }
  if (nx == 0 || (nz == 0 && !(ps.nz_global > 0))) return SBO_OK;
  SBO_TRY(sbo_ensure(ctx, ctx->pairctr, 2 * sizeof(unsigned long long)));
  SBO_CUDA(cudaMemsetAsync(ctx->pairctr.p, 0, 2 * sizeof(unsigned long long), ctx->stream));
  unsigned long long* ctr = (unsigned long long*)ctx->pairctr.p;
  const double* xc = (const double*)ctx->xs_pay.p; const double* ucb = xc + (size_t)d * nx; const double* thr = ucb + (size_t)nc * nx;
  const double* xn = (const double*)ctx->aux_x.p; const double* ax = xn + (size_t)d * nx; const double* bx = ax + (size_t)nc * nx;
  if (ps.mode == SBO_MODE_LIPSCHITZ) {
    PairConsts pc{};
    pc.nc = nc; pc.beta = ps.beta;
    for (int c = 0; c < nc; ++c) pc.L[c] = ps.L[c];
    // sharded SafeOpt expander: ALL unsafe points in grid order (sbo_pairs_set_global_unsafe_dev), this rank's share
    // of the candidate tiles; GoOSE target and single-GPU runs: the local unsafe points, every candidate
    // sharded GoOSE target with the all-gathered unsafe set: this rank's share of the (grid-ordered, compact) z tiles against
    // every candidate; result_dev then holds nc x nz_global flags indexed by the position in the global unsafe list
    const bool by_cand = ps.nz_global >= 0;
    const double* zc = (const double*)(by_cand ? ctx->gz_pay.p : ctx->zs_pay.p);
    const long long nzr = by_cand ? ps.nz_global : nz;
    const int stride = by_cand ? ps.seg_n : 1, off = by_cand ? ps.seg_rank : 0;
    const int* out_pos = (!goose && ps.canon) ? (const int*)ctx->perm_x.p : nullptr;
    unsigned char* hits = (unsigned char*)result_dev;
    if (nzr == 0) return SBO_OK;
    ev_begin(ctx, 4);
    SBO_TRY((with_int<1, SBO_MAX_D>(d, [&](auto D) {
      return launch_pairs<D>(ctx, goose, pc, nx, nzr, xc, ucb, thr, zc, hits, ctr, stride, off, out_pos);
    })));
    SBO_LAUNCH_CHECK();
    ev_end(ctx);
    ps.counted = true;
  } else {
    FantasyConsts fc{};
    fc.nc = nc; fc.d = d; fc.npad = ms.npad; fc.kernel = ms.kernel; fc.beta = ps.beta;
    for (int c = 0; c < nc; ++c) {
      fc.sf2[c] = ms.sf2[c + 1]; fc.sn2[c] = ms.sn2[c + 1];
      for (int k = 0; k < d; ++k) fc.inv_ell[c][k] = ms.inv_ell[c + 1][k];
    }
    const long long nxp = cdiv(nx, 256) * 256, nzp = cdiv(nz, 256) * 256;
    const double* zn = (const double*)ctx->aux_z.p; const double* mz = zn + (size_t)d * nz; const double* sz = mz + (size_t)nc * nz;
    int* cnt = goose ? nullptr : (int*)result_dev;
    uint32_t* hitw = goose ? (uint32_t*)result_dev : nullptr;    // GoOSE target: column OR instead of per-candidate counts
    const double* key_x = ps.sorted ? (const double*)ctx->key_x.p : nullptr;
    const double* key_z = ps.sorted ? (const double*)ctx->key_z.p : nullptr;
    const int* row_perm = ps.sorted ? (const int*)ctx->perm_x.p : nullptr;
    if (ps.precision == SBO_PREC_FP64 && ctx->opt_fantasy_f64_variant == 1) {
      // FP64 tensor cores (DMMA): 128 x 64 tiles over the exact-pruning item list
      DmmaArgs da{};
      da.nx = nx; da.nz = nz; da.nxp = nxp; da.nzp = nzp; da.np = ms.npad;
      da.nxt = (int)cdiv(nx, FD_BM); da.nzt = (int)cdiv(nz, FD_BN); da.gx = 32;
      da.Vx = (const double*)ctx->vx.p; da.Vz = (const double*)ctx->vz.p;
      da.xn = xn; da.ax = ax; da.bx = bx; da.zn = zn; da.mz = mz; da.sz = sz;
      da.counts = cnt; da.row_perm = row_perm; da.hit_words = hitw;
      da.n_items = cdiv(da.nxt, da.gx) * da.gx * (long long)da.nzt;
      ev_begin(ctx, 6);
      if (key_x && key_z) SBO_TRY(fantasy_build_items(ctx, nx, nz, FD_BM, FD_BN, da.gx, key_x, key_z, &da.item_list, &da.n_items));
      ev_end(ctx);
      SBO_REQUIRE(da.n_items < 2147483647LL, "too many tile pairs for one launch");
      const int RC = d + 2 * nc;
      const size_t smem = sizeof(double) * ((size_t)FD_STAGES * FD_STAGE_D + (size_t)(FD_BM + FD_BN) * RC);
      ev_begin(ctx, 4);
      if (da.n_items > 0) {
        SBO_TRY((with_int<1, SBO_MAX_D>(d, [&](auto D) { return with_flag(hitw != nullptr, [&](auto T) {
          return with_kernel(fc.kernel, [&](auto kc) -> int {
            SBO_CUDA(cudaFuncSetAttribute(k_fantasy_dmma<D, T, decltype(kc)>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_fantasy_dmma<D, T, decltype(kc)><<<(unsigned)da.n_items, 256, smem, ctx->stream>>>(fc, da);
            return SBO_OK;
          }); }); })));
        SBO_LAUNCH_CHECK();
      }
      ps.pairs_evaluated = da.n_items * (long long)FD_BM * FD_BN * nc;
    } else if (ps.precision == SBO_PREC_FP64) {
      dim3 grid((unsigned)cdiv(nz, FB), (unsigned)cdiv(nx, FB));

      SBO_REQUIRE(grid.y <= 65535, "too many candidates for the FP64 fantasy kernel");
      ev_begin(ctx, 4);
      with_int<1, SBO_MAX_D>(d, [&](auto D) { with_flag(hitw != nullptr, [&](auto T) { with_kernel(fc.kernel, [&](auto kc) {
        k_fantasy_f64<D, T, decltype(kc)><<<grid, 256, 0, ctx->stream>>>(fc, nx, nz, nxp, nzp, (const double*)ctx->vx.p,
            (const double*)ctx->vz.p, xn, ax, bx, zn, mz, sz, cnt, key_x, key_z, row_perm, ctr, hitw);
      }); }); });
      SBO_LAUNCH_CHECK();
      ps.counted = true;          // pairs evaluated = ctr[0] * nc (read back in finish)
      ps.count_scale = nc;
    } else {   // record prep is logged as phase 6, the GEMM kernel as phase 4 (begun inside)
      long long run_pairs = nx * nz;
      FantasyPruneArgs pr{key_x, key_z, row_perm, &run_pairs, 0, nullptr, nullptr, 0, nullptr, hitw, nullptr};
      const bool refine = (ps.precision == SBO_PREC_TF32X3 && ctx->opt_fantasy_refine >= 1) || (ps.precision == SBO_PREC_TF32 && ctx->opt_fantasy_refine >= 2);
      const bool bounds = refine && ctx->opt_fantasy_refine == 3;
      ps.bounds = bounds; ps.n_ambiguous = 0; ps.n_refined_safe = 0;
      if (bounds) {
        // bounds mode: no list and no FP64 pass.  counts = the pairs the error bound SETTLES as newly safe (a lower bound of the
        // FP64 counts), amb_rows = per candidate the number of pairs it cannot settle (counts + amb_rows is an upper bound).
        // GoOSE target: the hit words hold the z with a settled pair, amb_rows the words of the z with a pair inside the bound
        const size_t amb_b = goose ? sizeof(uint32_t) * (size_t)cdiv(nz, 32) : sizeof(int) * (size_t)nx;
        SBO_TRY(sbo_ensure(ctx, ctx->amb_rows, amb_b));
        SBO_CUDA(cudaMemsetAsync(ctx->amb_rows.p, 0, amb_b, ctx->stream));
        SBO_TRY(sbo_ensure(ctx, ctx->amb_ctr, 2 * sizeof(unsigned long long)));
        SBO_CUDA(cudaMemsetAsync(ctx->amb_ctr.p, 0, 2 * sizeof(unsigned long long), ctx->stream));
        pr.refine = 1; pr.amb_list = nullptr; pr.amb_cap = 0; pr.amb_count = (unsigned long long*)ctx->amb_ctr.p;
        if (goose) pr.amb_words = (uint32_t*)ctx->amb_rows.p;
        else pr.amb_rows = (int*)ctx->amb_rows.p;
      } else if (refine) {
        // list capacity: a 256th of the pairs, between 1 M and 32 M entries (C4: ~1 M ambiguous pairs of 3e10)
        long long cap = nx * nz / 256;
        cap = cap < (1LL << 20) ? (1LL << 20) : (cap > (1LL << 25) ? (1LL << 25) : cap);
        if (ctx->opt_fantasy_refine_cap > 0) cap = ctx->opt_fantasy_refine_cap;      // test hook: force the overflow path
        SBO_TRY(sbo_ensure(ctx, ctx->amb_list, sizeof(int2) * (size_t)cap));
        SBO_TRY(sbo_ensure(ctx, ctx->amb_ctr, 2 * sizeof(unsigned long long)));
        SBO_CUDA(cudaMemsetAsync(ctx->amb_ctr.p, 0, 2 * sizeof(unsigned long long), ctx->stream));
        pr.refine = 1; pr.amb_list = (int2*)ctx->amb_list.p; pr.amb_count = (unsigned long long*)ctx->amb_ctr.p;
        pr.amb_cap = ctx->opt_fantasy_refine_cap > 0 ? cap : (long long)(ctx->amb_list.cap / sizeof(int2));
      }
      SBO_TRY(fantasy_tc_run(ctx, fc, ps.precision == SBO_PREC_TF32X3 ? 1 : 0, nx, nz, nxp, nzp, (const float*)ctx->vx.p,
                             (const float*)ctx->vz.p, (const double*)ctx->aux_x.p, (const double*)ctx->aux_z.p, cnt, &pr));
      ps.pairs_evaluated = (ps.sorted ? run_pairs : nx * nz) * nc;
      if (bounds) {
        unsigned long long n_amb = 0;
        SBO_CUDA(cudaMemcpyAsync(&n_amb, ctx->amb_ctr.p, sizeof(n_amb), cudaMemcpyDeviceToHost, ctx->stream));
        SBO_CUDA(cudaStreamSynchronize(ctx->stream));
        ps.n_ambiguous = (long long)n_amb;
      } else if (refine) {
        // the list was sized by a heuristic: if more pairs were ambiguous than it holds (the entries past the capacity were
        // dropped, the counter kept counting), size it exactly and run the GEMM once more -- never refine a truncated list
        unsigned long long n_amb = 0;
        SBO_CUDA(cudaMemcpyAsync(&n_amb, ctx->amb_ctr.p, sizeof(n_amb), cudaMemcpyDeviceToHost, ctx->stream));
        SBO_CUDA(cudaStreamSynchronize(ctx->stream));
        if ((long long)n_amb > pr.amb_cap) {
          SBO_REQUIRE(n_amb < (1ULL << 31), "split/TF32 refinement: more than 2^31 ambiguous pairs on this shard (use fantasy_refine = 0 or fp64)");
          SBO_TRY(sbo_ensure(ctx, ctx->amb_list, sizeof(int2) * (size_t)n_amb));
          pr.amb_list = (int2*)ctx->amb_list.p; pr.amb_cap = (long long)(ctx->amb_list.cap / sizeof(int2));
          SBO_CUDA(cudaMemsetAsync(ctx->amb_ctr.p, 0, 2 * sizeof(unsigned long long), ctx->stream));
          SBO_CUDA(cudaMemsetAsync(result_dev, 0, res_bytes, ctx->stream));
          ev_end(ctx);
          SBO_TRY(fantasy_tc_run(ctx, fc, ps.precision == SBO_PREC_TF32X3 ? 1 : 0, nx, nz, nxp, nzp, (const float*)ctx->vx.p,
                                 (const float*)ctx->vz.p, (const double*)ctx->aux_x.p, (const double*)ctx->aux_z.p, cnt, &pr));
        }
        ev_end(ctx);
        ev_begin(ctx, 7);
        SBO_TRY(refine_ambiguous(ctx, fc, nx, nz, cnt, row_perm, hitw));
      }
    }
    ev_end(ctx);
  }
  return SBO_OK;
}

// GoOSE fantasy target: hit bits over the prepared z slots -> grid-ordered target mask; bounds mode: slots with an ambiguous
// pair and no settled one -> undecided mask
__global__ void __launch_bounds__(256)
k_slots_to_mask(long long n, const long long* __restrict__ idx, const uint32_t* __restrict__ hit, const uint32_t* __restrict__ amb,
                uint32_t* __restrict__ mask, uint32_t* __restrict__ und) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const long long p = idx[t];
  const uint32_t bit = 1u << (t & 31);
  if (hit[t >> 5] & bit) atomicOr(mask + (p >> 5), 1u << (p & 31));
  else if (amb && (amb[t >> 5] & bit)) atomicOr(und + (p >> 5), 1u << (p & 31));
}

// result_dev: the (all-reduced) per-candidate results; the local candidates are rows [offset, offset+nx_local).
// GoOSE fantasy target: the local hit words of pairs_run (no reduction needed: every rank paired all candidates)
int pairs_finish(sbo_ctx* ctx, int goose, long long offset, const void* result_dev, sbo_pair_result* out, int32_t* counts_host) {
  PairStage& ps = ctx->ps;
  SBO_REQUIRE(ps.prepared && ps.imported, "sbo_pairs_finish: run the pair stage first");
  SBO_REQUIRE(out != nullptr, "null result");
  const ModelSpec& ms = ctx->ms;
  const int nc = ms.G - 1;
  const long long count = ctx->gs.count, nw = mask_words(ctx);
  const long long nx = ps.nx_local, nz = ps.nz_local, nxt = ps.nx_total;
  const bool fantasy = ps.mode == SBO_MODE_FANTASY;
  const bool counted = fantasy && !goose;              // per-candidate newly-safe counts (fantasy expander)
  SBO_REQUIRE(goose || (offset >= 0 && offset + nx <= nxt), "local candidate slice out of range");
  memset(out, 0, sizeof(*out));
  out->best_idx = -1;
  out->best_value = goose ? INFINITY : -INFINITY;
  for (int c = 0; c < SBO_MAX_G; ++c) { out->per_idx[c] = -1; out->per_value[c] = goose ? INFINITY : -INFINITY; }
  out->n_x = nxt; out->n_z = ps.nz_full;                 // |Z| of the local shard; nz = what was actually paired
  out->pairs_algorithmic = nxt * ps.nz_full * nc;
  const int nmask = fantasy ? 1 : nc;
  DevBuf& mbuf = goose ? ctx->m_tgt : ctx->m_exp;
  SBO_TRY(sbo_ensure(ctx, mbuf, sizeof(uint32_t) * (size_t)(nc > 0 ? nc : 1) * nw));
  SBO_CUDA(cudaMemsetAsync(mbuf.p, 0, sizeof(uint32_t) * (size_t)(nc > 0 ? nc : 1) * nw, ctx->stream));
  SBO_TRY(sbo_ensure(ctx, ctx->pairctr, 2 * sizeof(unsigned long long)));
  if (counted) {
    SBO_TRY(sbo_ensure(ctx, ctx->counts, sizeof(int) * (size_t)count));
    SBO_CUDA(cudaMemsetAsync(ctx->counts.p, 0, sizeof(int) * (size_t)count, ctx->stream));
  }
  unsigned long long h[2] = {0, 0};
  const long long nloc = goose ? nz : nx;
  const bool have = nc > 0 && nloc > 0 && nxt > 0 && (fantasy || nz > 0 || (!goose && ps.nz_global > 0)) && result_dev != nullptr;
  const bool bounds = fantasy && ps.bounds && have;
  unsigned long long h_und = 0;
  if (have) {
    ev_begin(ctx, 6);
    const long long* idx = (const long long*)(goose ? ctx->zs_idx.p : ctx->xs_idx.p);
    if (bounds) {
      SBO_TRY(sbo_ensure(ctx, ctx->m_und, sizeof(uint32_t) * (size_t)nw));
      SBO_CUDA(cudaMemsetAsync(ctx->m_und.p, 0, sizeof(uint32_t) * (size_t)nw, ctx->stream));
    }
    if (fantasy && goose)
      k_slots_to_mask<<<(unsigned)cdiv(nz, 256), 256, 0, ctx->stream>>>(nz, idx, (const uint32_t*)result_dev, bounds ? (const uint32_t*)ctx->amb_rows.p : nullptr,
                                                                       (uint32_t*)mbuf.p, (uint32_t*)ctx->m_und.p);
    else if (fantasy)
      k_counts_scatter<<<(unsigned)cdiv(nx, 256), 256, 0, ctx->stream>>>(nx, offset, idx, (const int*)result_dev, (int*)ctx->counts.p, (uint32_t*)mbuf.p);
    else
      k_hits_to_mask<<<(unsigned)cdiv(nloc, 256), 256, 0, ctx->stream>>>(nc, nloc, goose ? nz : nxt, goose ? 0 : offset, idx,
                                                                          (const unsigned char*)result_dev, (uint32_t*)mbuf.p, nw);
    SBO_LAUNCH_CHECK();
    unsigned long long* ctr = (unsigned long long*)ctx->pairctr.p;
    SBO_CUDA(cudaMemsetAsync(ctr + 1, 0, sizeof(unsigned long long), ctx->stream));
    k_union_count<<<(unsigned)cdiv(nw, 256), 256, 0, ctx->stream>>>(nmask, (const uint32_t*)mbuf.p, nw, ctr + 1);
    SBO_LAUNCH_CHECK();
    SBO_CUDA(cudaMemcpyAsync(h, ctr, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    if (bounds) {
      // amb_rows holds the (all-reduced, sbo_*_step_sharded) per-candidate ambiguous-pair counts in the layout of result_dev
      // (GoOSE target: the undecided mask was built above from the local ambiguous words)
      if (!goose) {
        k_undecided_mask<<<(unsigned)cdiv(nx, 256), 256, 0, ctx->stream>>>(nx, offset, idx, (const int*)result_dev, (const int*)ctx->amb_rows.p,
                                                                            (int*)ctx->counts.p, (uint32_t*)ctx->m_und.p);
        SBO_LAUNCH_CHECK();
      }
      SBO_CUDA(cudaMemsetAsync(ctr + 1, 0, sizeof(unsigned long long), ctx->stream));
      k_union_count<<<(unsigned)cdiv(nw, 256), 256, 0, ctx->stream>>>(1, (const uint32_t*)ctx->m_und.p, nw, ctr + 1);
      SBO_LAUNCH_CHECK();
      SBO_CUDA(cudaMemcpyAsync(&h_und, ctr + 1, sizeof(h_und), cudaMemcpyDeviceToHost, ctx->stream));
    }
    ev_end(ctx);
  }
  if (counts_host) {
    if (counted) SBO_CUDA(cudaMemcpyAsync(counts_host, ctx->counts.p, sizeof(int32_t) * (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
    else memset(counts_host, 0, sizeof(int32_t) * (size_t)count);
  }
  SBO_CUDA(cudaStreamSynchronize(ctx->stream));
  ev_collect(ctx);
  out->n_hit = (int64_t)h[1];
  out->n_ambiguous = ps.n_ambiguous; out->n_refined_safe = ps.n_refined_safe;
  out->n_undecided = bounds ? (int64_t)h_und : 0;
  out->undecided_best_idx = -1; out->undecided_best_value = goose ? INFINITY : -INFINITY;
  if (ps.counted) out->pairs_evaluated = (int64_t)h[0] * ps.count_scale;
  else out->pairs_evaluated = ps.pairs_evaluated;
  if (out->pairs_evaluated > out->pairs_algorithmic) out->pairs_evaluated = out->pairs_algorithmic;
  // the expander (target) masks are complete: a batch acquisition may start from them
  stage_changed(ctx, goose ? Change::TARGET : Change::EXPANDER);
  if (!have) return SBO_OK;
  // per-constraint arg-reduction, then first-best across constraints (SafeOpt.py:120-122 / GoOSE.py:110-112)
  const double keep5 = ctx->phase_ms[5];
  double acc5 = 0.0;
  for (int c = 0; c < nmask; ++c) {
    int64_t idx; double val;
    SBO_TRY(argreduce_run(ctx, goose ? SBO_ARGMIN_LCB0 : SBO_ARGMAX_VAR0, (const uint32_t*)mbuf.p + (size_t)c * nw, nullptr, &idx, &val));
    acc5 += ctx->phase_ms[5];
    out->per_idx[c] = idx; out->per_value[c] = val;
    if (idx >= 0) {
      const bool better = out->best_idx < 0 || (goose ? (val < out->best_value) : (val > out->best_value));
      if (better) { out->best_idx = idx; out->best_value = val; }
    }
  }
  if (bounds && out->n_undecided > 0) {
    SBO_TRY(argreduce_run(ctx, goose ? SBO_ARGMIN_LCB0 : SBO_ARGMAX_VAR0, (const uint32_t*)ctx->m_und.p, nullptr, &out->undecided_best_idx,
                          &out->undecided_best_value));
    acc5 += ctx->phase_ms[5];
  }
  ctx->phase_ms[5] = keep5 + acc5;
  return SBO_OK;
}

// ---------------------------------------------------------------------------------------------
// single-GPU compositions used by sbo_expander / sbo_goose_target: import the context's own export
// ---------------------------------------------------------------------------------------------
static int pairs_single(sbo_ctx* ctx, int mode, int precision, bool goose, double beta, const double* L,
                        sbo_pair_result* out, int32_t* counts_host) {
  SBO_REQUIRE(out != nullptr, "null result");
  sbo_pairs_info info;
  SBO_TRY(pairs_prepare(ctx, mode, precision, beta, L, &info));
  const long long nx = info.n_x_local, nz = info.n_z_local;
  const int nc = ctx->ms.G - 1;
  SBO_TRY(sbo_ensure(ctx, ctx->exp_rows, sizeof(double) * (size_t)(nx > 0 ? nx : 1) * info.row_doubles));
  if (mode == SBO_MODE_FANTASY) SBO_TRY(sbo_ensure(ctx, ctx->exp_v, (size_t)(nx > 0 ? nx : 1) * info.vrow_bytes));
  SBO_TRY(pairs_export(ctx, ctx->exp_rows.p, ctx->exp_v.p));
  SBO_TRY(pairs_import(ctx, nx, ctx->exp_rows.p, ctx->exp_v.p));
  const size_t res_bytes = (mode == SBO_MODE_FANTASY) ? (goose ? sizeof(uint32_t) * (size_t)cdiv(nz, 32) : sizeof(int) * (size_t)nx)
                                                     : (size_t)(nc > 0 ? nc : 1) * (goose ? nz : nx);
  SBO_TRY(sbo_ensure(ctx, ctx->hits, res_bytes));
  SBO_TRY(pairs_run(ctx, goose ? 1 : 0, ctx->hits.p));
  return pairs_finish(ctx, goose ? 1 : 0, 0, ctx->hits.p, out, counts_host);
}

int pairs_lipschitz(sbo_ctx* ctx, bool goose, double beta, const double* L, sbo_pair_result* out) {
  SBO_REQUIRE(L != nullptr, "Lipschitz constants required");
  return pairs_single(ctx, SBO_MODE_LIPSCHITZ, SBO_PREC_FP64, goose, beta, L, out, nullptr);
}

int pairs_fantasy(sbo_ctx* ctx, int precision, double beta, sbo_pair_result* out, int32_t* counts_host) {
  return pairs_single(ctx, SBO_MODE_FANTASY, precision, false, beta, nullptr, out, counts_host);
}

int pairs_goose_fantasy(sbo_ctx* ctx, int precision, double beta, sbo_pair_result* out) {
  return pairs_single(ctx, SBO_MODE_FANTASY, precision, true, beta, nullptr, out, nullptr);
}
