// fantasy_tc.cu -- TF32 tcgen05/TMEM fantasy-expander GEMM for sm_100a (north_star "Expanders" bullet;
// SURVEY.md section 8 row a12; not in the reference).
//
//   for every candidate x (rows, MMA M = 128) and every unsafe z (columns, MMA N = BN) and every constraint GP c:
//       acc  = v_x . v_z                         tcgen05.mma kind::tf32, FP32 accumulator in TMEM, K = npad
//       cov  = k_c(z,x) - acc                    covariance recomputed in the epilogue (SE: ex2.approx; Matern:
//                                                sqrt.approx + ex2.approx + polynomial, common.cuh)
//       mu'  = m_z + cov * a_x ,  s2' = s_z - cov^2 * b_x     (rank-1 fantasy update, normalised units)
//       ok  &= mu' >= 0  &&  mu'^2 >= beta^2 * s2'            (<=> mu' - beta*sqrt(max(s2',0)) >= 0)
//   g(x) = popcount over z of ok  -> atomicAdd per candidate.
//
// Structure (one persistent CTA per SM, 256 threads):
//   warp 0   TMA producer: 3-D tensor maps over Vx[c][row][k] / Vz[c][row][k], 128-byte swizzled boxes of
//            32 TF32 columns, STAGES-deep smem ring (full/empty mbarriers)
//   warp 1   MMA issuer: one elected lane issues 4 x (M128,N=BN,K8) tcgen05.mma per stage; tcgen05.commit
//            releases the smem stage and, after the last K block, publishes the TMEM accumulator slot
//   warp 2   TMEM allocator (512 columns = 512/BN accumulator slots), then work-item scheduler
//   warp 3   column-record loader: per (z tile, constraint) unit one cp.async.bulk of BN records into smem
//   warps 4-7 epilogue: tcgen05.ld 32x32b.x32 -> registers, fused kernel/rank-1/threshold math, per-row
//            bitmask AND across constraints, popcount into a per-thread counter.
// A "unit" is (tile pair, constraint); TMEM slots form a ring over units so the epilogue of unit u overlaps the
// MMAs of unit u+1.  Work items = (x tile, z tile) pairs handed out dynamically by warp 2 (atomic counter -> smem
// ring) in an order that keeps a group of x tiles L2-resident while the z tiles stream past.
#include "common.cuh"
#include <cuda.h>
#include <math.h>

namespace tc {

constexpr int BM = 128;        // candidates per tile (MMA M, TMEM lanes)
constexpr int BK = 32;         // TF32 elements per smem row = 128 bytes = one SWIZZLE_128B atom
constexpr int UK = 8;          // K per tcgen05.mma kind::tf32
constexpr int GX = 37;         // x tiles per raster group (4 z chunks in flight on 148 SMs)

struct Params {
  int nc, kblocks, nkb, npad, split, nxt, nzt;   // kblocks = split ? 3*nkb : nkb
  int gx;                                        // x tiles per raster group (2-CTA kernel; the 1-CTA kernel uses GX)
  long long nx, nz, nxp, nzp, n_items;
  const float* rowrec;   // [nc][nxp][RS]
  const float* colrec;   // [nc][nzp][RS]
  int* counts;           // [nx]
  int* err;
  unsigned int* sched_counter;   // zeroed before every launch
  const long long* item_list;    // feasible raster items in ascending order (exact pruning), or null = all n_items
  const int* row_perm;           // sorted candidate slot -> row of `counts` (null = identity)
  // refinement (REFINE kernels): pairs whose decision the FP32 error bound cannot settle are NOT counted here but
  // appended as (candidate slot, z column) to amb_list for the FP64 re-evaluation (pairs.cu k_refine_pairs)
  int2* amb_list;
  unsigned long long* amb_count;   // [0] entries appended (may exceed the capacity: overflow is detected by the host)
  long long amb_cap;
  int* amb_rows;                   // bounds mode (fantasy_refine = 3): per-candidate number of ambiguous pairs, no list
  float e_abs, d_mu, d_t;          // absolute error terms of the FP32 epilogue (covariance, mean, variance side)
  // GoOSE target (2-CTA kernel only; counts unused): bit z of hit_words is set when some valid candidate row makes column z
  // safe; bounds mode sets bit z of amb_words instead of amb_rows when column z has a pair inside the error bound
  uint32_t* hit_words;
  uint32_t* amb_words;
  int kernel;                      // enum sbo_kernel; Matern: sf2 of every constraint (SE carries it in the row records)
  float ksf2[SBO_MAX_G - 1];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err, int tag) {
  if (mbar_try(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try(bar, parity)) {
    if (clock64() - t0 > 8000000000LL) {
      if (err) atomicExch(err, tag);
      __trap();
    }
  }
}

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 "version 1"): 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// w |= bit  iff  mu >= 0 and mu^2 >= t   (two FSETP chained through the predicate + one predicated LOP3)
__device__ __forceinline__ void set_bit_if_safe(uint32_t& w, float mu, float mm, float t, uint32_t bit) {
  asm("{\n\t.reg .pred p;\n\t"
      "setp.ge.f32 p, %1, 0f00000000;\n\t"
      "setp.ge.and.f32 p, %2, %3, p;\n\t"
      "@p or.b32 %0, %0, %4;\n\t}"
      : "+r"(w)
      : "f"(mu), "f"(mm), "f"(t), "r"(bit));
}

// row constants of one candidate for one constraint, duplicated into both halves of a packed pair
template <int D4>
struct RowConsts {
  uint64_t xx[4 * D4], Cx, ax, nbx, ex;      // ex: sqrt(c1)*|v_x| (refinement band), duplicated like the others
  uint64_t kf;                               // Matern: (sf2_c, sf2_c); unused by SE
  __device__ __forceinline__ void load(const float* __restrict__ rowrec_row) {
    const float4* rr = reinterpret_cast<const float4*>(rowrec_row);
#pragma unroll
    for (int v = 0; v < D4; ++v) {
      const float4 t = __ldg(rr + v);
      xx[4 * v] = pk2(t.x, t.x); xx[4 * v + 1] = pk2(t.y, t.y); xx[4 * v + 2] = pk2(t.z, t.z); xx[4 * v + 3] = pk2(t.w, t.w);
    }
    const float4 rt = __ldg(rr + D4);
    Cx = pk2(rt.x, rt.x); ax = pk2(rt.y, rt.y); nbx = pk2(-rt.z, -rt.z); ex = pk2(rt.w, rt.w);
  }
};

// One 32-column chunk of the fused epilogue for one candidate row: acc[32] = v_x . v_z from TMEM, `rec` = the 16
// pair-interleaved column records of the chunk in shared memory ((4*D4+4) float2 per column pair:
// z_k pairs, -Bz pair, m_z pair, s'_z pair, pad).  Same operations in the same order as the scalar form
// (e = (Cx - Bz) + sum xx_k z_k; cov = k(e) - acc; mu = cov*a + m; t = s' - cov^2 b'), two columns per FFMA2.
// k(e) is KC::value_f32x2 (common.cuh): exp2(e) for SE, sf2 P(t) exp(-t) with t = sqrt(-e) for Matern.
template <int D4, class KC>
__device__ __forceinline__ uint32_t epilogue_chunk(const uint32_t (&acc)[32], const uint64_t* __restrict__ rec, const RowConsts<D4>& rc,
                                                   const KC& kc) {
  constexpr int RS = 4 * D4 + 4;
  const uint64_t minus1 = pk2(-1.f, -1.f);
  uint32_t w = 0;
#pragma unroll
  for (int jp = 0; jp < 16; ++jp) {
    const uint64_t* p = rec + jp * RS;
    uint64_t e = add2(rc.Cx, p[4 * D4]);
#pragma unroll
    for (int k = 0; k < 4 * D4; ++k) e = fma2(rc.xx[k], p[k], e);
    const uint64_t ex = kc.value_f32x2(e, rc.kf);
    const uint64_t a2 = pk2(__uint_as_float(acc[2 * jp]), __uint_as_float(acc[2 * jp + 1]));
    const uint64_t cov = fma2(a2, minus1, ex);
    const uint64_t mu = fma2(cov, rc.ax, p[4 * D4 + 1]);
    const uint64_t t = fma2(mul2(cov, cov), rc.nbx, p[4 * D4 + 2]);
    const uint64_t mm = mul2(mu, mu);
    float mu0, mu1, t0, t1, m0, m1;
    upk2(mu, mu0, mu1); upk2(t, t0, t1); upk2(mm, m0, m1);
    set_bit_if_safe(w, mu0, m0, t0, 1u << (2 * jp));
    set_bit_if_safe(w, mu1, m1, t1, 2u << (2 * jp));
  }
  return w;
}

// Refining variant.  E = ex*ez + e_abs bounds the error of the computed covariance (operand rounding / split, one ulp
// of the running sum per tensor-core accumulation step, ex2.approx, FP32 records); d_mu / d_t bound the FP32 rounding of
// the mean and variance sides of the test.  The updated bound f(cov) = mu' - beta*sigma' is CONVEX in cov, satisfies
// f(-c) <= f(c) (a_x >= 0) and increases for cov >= 0, so over the interval [cov - E, cov + E] it is bounded by
// f(|cov| + E):
//   U (settled unsafe)  <=  f(|cov| + E) < 0 evaluated OPTIMISTICALLY (+d_mu, -d_t)               -- ONE evaluation
//   S (settled safe)    <=  cov - E >= 0 (monotone branch) and f(cov - E) >= 0 evaluated PESSIMISTICALLY (-d_mu, +d_t);
//                           only needed where U fails: whole warps skip it (almost every pair is settled unsafe).
// Everything else is AMBIGUOUS and goes to the FP64 re-evaluation (pairs.cu refine_ambiguous).
template <int D4, class KC>
__device__ __forceinline__ void epilogue_chunk_refine(const uint32_t (&acc)[32], const uint64_t* __restrict__ rec, const RowConsts<D4>& rc,
                                                      const KC& kc, uint64_t e_abs2, uint64_t d_mu2, uint64_t d_t2, uint32_t& S,
                                                      uint32_t& U) {
  constexpr int RS = 4 * D4 + 4;
  const uint64_t minus1 = pk2(-1.f, -1.f);
  uint32_t wup = 0, wsf = 0;
#pragma unroll
  for (int jp = 0; jp < 16; ++jp) {
    const uint64_t* p = rec + jp * RS;
    uint64_t e = add2(rc.Cx, p[4 * D4]);
#pragma unroll
    for (int k = 0; k < 4 * D4; ++k) e = fma2(rc.xx[k], p[k], e);
    const uint64_t ex = kc.value_f32x2(e, rc.kf);
    const uint64_t a2 = pk2(__uint_as_float(acc[2 * jp]), __uint_as_float(acc[2 * jp + 1]));
    const uint64_t cov = fma2(a2, minus1, ex);
    const uint64_t E = fma2(rc.ex, p[4 * D4 + 3], e_abs2);                // ex*ez + e_abs
    float c0, c1, E0, E1;
    upk2(cov, c0, c1); upk2(E, E0, E1);
    const uint64_t h = pk2(fabsf(c0) + E0, fabsf(c1) + E1);               // |cov| + E (the abs is an operand modifier)
    const uint64_t m_opt = add2(p[4 * D4 + 1], d_mu2);                    // m_z + d_mu
    const uint64_t s_opt = fma2(d_t2, minus1, p[4 * D4 + 2]);             // s'_z - d_t
    const uint64_t mu_h = fma2(h, rc.ax, m_opt);
    const uint64_t t_h = fma2(mul2(h, h), rc.nbx, s_opt);
    const uint64_t mm_h = mul2(mu_h, mu_h);
    float a0, a1, b0, b1, q0, q1;
    const uint32_t pairbits = 3u << (2 * jp);
    upk2(mu_h, a0, a1); upk2(t_h, b0, b1); upk2(mm_h, q0, q1);
    set_bit_if_safe(wup, a0, q0, b0, 1u << (2 * jp)); set_bit_if_safe(wup, a1, q1, b1, 2u << (2 * jp));
    if (__any_sync(0xffffffffu, (wup & pairbits) != 0u)) {                // warp-uniform: some pair here is not settled unsafe
      const uint64_t cl = fma2(E, minus1, cov);
      const uint64_t m_pes = fma2(d_mu2, minus1, p[4 * D4 + 1]), s_pes = add2(p[4 * D4 + 2], d_t2);   // m_z - d_mu, s'_z + d_t
      const uint64_t mu_sf = fma2(cl, rc.ax, m_pes), t_sf = fma2(mul2(cl, cl), rc.nbx, s_pes), mm_sf = mul2(mu_sf, mu_sf);
      float l0, l1;
      upk2(mu_sf, a0, a1); upk2(t_sf, b0, b1); upk2(mm_sf, q0, q1); upk2(cl, l0, l1);
      a0 = l0 < 0.f ? l0 : a0; a1 = l1 < 0.f ? l1 : a1;                   // lo < 0: not on the monotone branch -> never "settled safe"
      set_bit_if_safe(wsf, a0, q0, b0, 1u << (2 * jp)); set_bit_if_safe(wsf, a1, q1, b1, 2u << (2 * jp));
    }
  }
  S = wsf;
  U = ~wup;
}

// work item = one (x tile, z tile) pair, all constraints.  Items are ordered so that a group of GX x tiles sweeps
// the z tiles together: the GX*768 KB of x operands stay L2-resident while each z tile is reused by GX consecutive
// items.  Items are handed out dynamically (atomic counter -> smem ring), which bounds the drift between CTAs to
// about one item and keeps that reuse window intact (a static round-robin let CTAs drift apart: ncu showed 44 % L2
// hit rate and 3 TB of DRAM reads for 5.4 GB of operands).
__device__ __forceinline__ bool item_coords(const Params& p, long long item, int& xt, int& zt) {
  const long long per_group = (long long)GX * p.nzt;
  const int xg = (int)(item / per_group);
  const int r = (int)(item % per_group);
  zt = r / GX;
  xt = xg * GX + r % GX;
  return xt < p.nxt;
}

constexpr int SCHED = 4;   // depth of the work-item ring

template <int BN, int D4>
struct Cfg {
  static constexpr int RS = 4 * D4 + 4;                 // floats per row/column record
  static constexpr int SLOTS = 512 / BN;                // TMEM accumulator slots
  static constexpr int STAGE_BYTES = (BM + BN) * 128;   // A tile + B tile
  static constexpr int STAGES = (BN == 128) ? 5 : 4;
  static constexpr int COL_BYTES = BN * RS * 4;
  static constexpr int NBARS = 2 * STAGES + 2 * SLOTS + 4 + 2 * SCHED;
  static constexpr int SMEM_BYTES = 1024 + STAGES * STAGE_BYTES + 2 * COL_BYTES + 8 * NBARS + 64;
};

template <int BN, int D4, int EW>   // EW = epilogue warps (4 or 8): 8 puts two warps on every scheduler and splits the columns
__global__ void __launch_bounds__(128 + 32 * EW, 1)
k_fantasy_tc(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const Params p) {
  using C = Cfg<BN, D4>;
  constexpr int RS = C::RS, SLOTS = C::SLOTS, STAGES = C::STAGES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;          // SWIZZLE_128B tiles need 1024 B alignment
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t tiles = base;
  const uint32_t colbuf = base + STAGES * C::STAGE_BYTES;
  const float* colbuf_ptr = reinterpret_cast<const float*>(base_ptr + STAGES * C::STAGE_BYTES);
  const uint32_t bars = colbuf + 2 * C::COL_BYTES;
  uint8_t* tail = base_ptr + STAGES * C::STAGE_BYTES + 2 * C::COL_BYTES + 8 * C::NBARS;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(tail);
  volatile int* sched_items = reinterpret_cast<volatile int*>(tail + 16);   // SCHED ints
  // barrier map (8 bytes each)
  auto bar_full = [&](int s) { return bars + 8 * s; };
  auto bar_empty = [&](int s) { return bars + 8 * (STAGES + s); };
  auto bar_tfull = [&](int s) { return bars + 8 * (2 * STAGES + s); };
  auto bar_tempty = [&](int s) { return bars + 8 * (2 * STAGES + SLOTS + s); };
  auto bar_cfull = [&](int b) { return bars + 8 * (2 * STAGES + 2 * SLOTS + b); };
  auto bar_cempty = [&](int b) { return bars + 8 * (2 * STAGES + 2 * SLOTS + 2 + b); };
  auto bar_sfull = [&](int s) { return bars + 8 * (2 * STAGES + 2 * SLOTS + 4 + s); };
  auto bar_sempty = [&](int s) { return bars + 8 * (2 * STAGES + 2 * SLOTS + 4 + SCHED + s); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_empty(s), 1); }
    for (int s = 0; s < SLOTS; ++s) { mbar_init(bar_tfull(s), 1); mbar_init(bar_tempty(s), EW); }
    for (int b = 0; b < 2; ++b) { mbar_init(bar_cfull(b), 1); mbar_init(bar_cempty(b), EW); }
    for (int s = 0; s < SCHED; ++s) { mbar_init(bar_sfull(s), 1); mbar_init(bar_sempty(s), 3 + EW); }   // 3 lanes + EW warps
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_holder;

  // every consumer role walks the same ring of work items
  int ss = 0; uint32_t sph = 0;
  // single-lane roles call it with warp_wide = false; the epilogue warps (all lanes read the slot) sync the warp
  // before lane 0 releases the slot
  auto next_item = [&](bool warp_wide) -> int {
    mbar_wait(bar_sfull(ss), sph, p.err, 7);
    const int item = sched_items[ss];
    if (warp_wide) __syncwarp();
    if (!warp_wide || lane == 0) mbar_arrive(bar_sempty(ss));
    if (++ss == SCHED) { ss = 0; sph ^= 1; }
    return item;
  };

  if (warp == 2) {
    // ================================ scheduler ================================
    if (lane == 0) {
      int s2 = 0; uint32_t ph2 = 0;
      for (;;) {
        long long item = (long long)atomicAdd(p.sched_counter, 1u);
        int v = (item < p.n_items) ? (p.item_list ? (int)p.item_list[item] : (int)item) : -1;
        mbar_wait(bar_sempty(s2), ph2 ^ 1, p.err, 8);
        sched_items[s2] = v;
        mbar_arrive(bar_sfull(s2));
        if (++s2 == SCHED) { s2 = 0; ph2 ^= 1; }
        if (v < 0) break;
      }
    }
  } else if (warp == 0) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (;;) {
        const int item = next_item(false);
        if (item < 0) break;
        int xt, zt;
        if (!item_coords(p, item, xt, zt)) continue;
        for (int c = 0; c < p.nc; ++c)
          for (int kb = 0; kb < p.kblocks; ++kb) {
            mbar_wait(bar_empty(stage), phase ^ 1, p.err, 1);
            mbar_expect_tx(bar_full(stage), C::STAGE_BYTES);
            const uint32_t sa = tiles + stage * C::STAGE_BYTES;
            // split-TF32 rows are [hi | lo]: K segments (x_hi,z_lo), (x_lo,z_hi), then (x_hi,z_hi).  The two small
            // cross terms are accumulated FIRST, while the FP32 accumulator is still ~2^-11 of its final size, so the
            // tensor core's per-step accumulation rounding (one ulp of the running sum) cannot swallow them.
            const int seg = p.split ? kb / p.nkb : 2, kk = (kb - (p.split ? seg : 0) * p.nkb) * BK;
            tma_load_3d(sa, &tmA, bar_full(stage), kk + (seg == 1 ? p.npad : 0), xt * BM, c);
            tma_load_3d(sa + BM * 128, &tmB, bar_full(stage), kk + (seg == 0 ? p.npad : 0), zt * BN, c);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    if (lane == 0) {
      constexpr uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      int stage = 0; uint32_t phase = 0;
      int slot = 0; uint32_t sphase = 0;
      for (;;) {
        const int item = next_item(false);
        if (item < 0) break;
        int xt, zt;
        if (!item_coords(p, item, xt, zt)) continue;
        for (int c = 0; c < p.nc; ++c) {
          mbar_wait(bar_tempty(slot), sphase ^ 1, p.err, 2);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t tmem_d = tmem_base + (uint32_t)(slot * BN);
          for (int kb = 0; kb < p.kblocks; ++kb) {
            mbar_wait(bar_full(stage), phase, p.err, 3);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t sa = tiles + stage * C::STAGE_BYTES;
            const uint64_t adesc = make_desc(sa), bdesc = make_desc(sa + BM * 128);
#pragma unroll
            for (int k = 0; k < BK / UK; ++k)
              mma_tf32(tmem_d, adesc + (uint64_t)(k * UK * 4 / 16), bdesc + (uint64_t)(k * UK * 4 / 16), idesc,
                       (kb | k) ? 1u : 0u);
            mma_commit(bar_empty(stage));                 // frees the smem stage when these MMAs retire
            if (kb == p.kblocks - 1) mma_commit(bar_tfull(slot));   // accumulator complete
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          if (++slot == SLOTS) { slot = 0; sphase ^= 1; }
        }
      }
    }
  } else if (warp == 3) {
    // ================================ column-record loader ================================
    if (lane == 0) {
      int b = 0; uint32_t bphase = 0;
      for (;;) {
        const int item = next_item(false);
        if (item < 0) break;
        int xt, zt;
        if (!item_coords(p, item, xt, zt)) continue;
        for (int c = 0; c < p.nc; ++c) {
          mbar_wait(bar_cempty(b), bphase ^ 1, p.err, 4);
          mbar_expect_tx(bar_cfull(b), C::COL_BYTES);
          bulk_load_1d(colbuf + b * C::COL_BYTES, p.colrec + ((size_t)c * p.nzp + (size_t)zt * BN) * RS, C::COL_BYTES,
                       bar_cfull(b));
          if (++b == 2) { b = 0; bphase ^= 1; }
        }
      }
    }
  } else {
    // ================================ epilogue (warps 4 .. 4+EW-1) ================================
    const int q = warp & 3;                       // TMEM lane quarter: a warp may touch lanes 32*(warp%4) .. +31
    const int half = (warp - 4) >> 2;             // EW = 8: warps 8-11 take the upper half of the columns
    constexpr int NCH = BN / 32 / (EW / 4);       // 32-column chunks per warp per unit
    const int row = q * 32 + lane;
    int slot = 0; uint32_t sphase = 0;
    int b = 0; uint32_t bphase = 0;
    for (;;) {
      const int item = next_item(true);
      if (item < 0) break;
      int xt, zt;
      if (!item_coords(p, item, xt, zt)) continue;
      const long long xrow = (long long)xt * BM + row;
      uint32_t bits[NCH];
#pragma unroll
      for (int h = 0; h < NCH; ++h) bits[h] = 0xffffffffu;
      for (int c = 0; c < p.nc; ++c) {
        // row record of this candidate for constraint c: xx[4*D4], Cx, a, b', pad
        RowConsts<D4> rc;
        rc.load(p.rowrec + ((size_t)c * p.nxp + xrow) * RS);
        mbar_wait(bar_cfull(b), bphase, p.err, 5);
        mbar_wait(bar_tfull(slot), sphase, p.err, 6);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // pair-interleaved column records: RS packed pairs per two columns
        const uint64_t* cb = reinterpret_cast<const uint64_t*>(colbuf_ptr + (size_t)b * BN * RS) + (size_t)half * NCH * 16 * RS;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(slot * BN + half * NCH * 32);
#pragma unroll
        for (int h = 0; h < NCH; ++h) {
          uint32_t r[32];
          tmem_ld32(taddr + h * 32, r);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          bits[h] &= epilogue_chunk<D4>(r, cb + (size_t)h * 16 * RS, rc, SE(SBO_KERNEL_SE));
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) { mbar_arrive(bar_tempty(slot)); mbar_arrive(bar_cempty(b)); }
        if (++slot == SLOTS) { slot = 0; sphase ^= 1; }
        if (++b == 2) { b = 0; bphase ^= 1; }
      }
      int cnt = 0;
#pragma unroll
      for (int h = 0; h < NCH; ++h) cnt += __popc(bits[h]);
      if (xrow < p.nx && cnt) atomicAdd(p.counts + (p.row_perm ? p.row_perm[xrow] : xrow), cnt);
    }
  }
  // ---- teardown
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// =============================================================================================
// 2-CTA variant (cta_group::2): a cluster of two CTAs on one TPC computes a 256 x 256 tile pair with ONE
// tcgen05.mma M=256 stream issued by the leader CTA (cluster rank 0).  Each CTA stages only its own half of both
// operands per K block -- 128 candidate rows (A half) + 128 unsafe rows (B half) = 32 KB instead of 48 KB -- so the
// L2->SM operand traffic per MMA drops by a third and the same shared memory holds 6 stages instead of 4.
// Each CTA's TMEM holds the accumulator rows of ITS 128 candidates for all 256 z columns; the epilogue is the
// 1-CTA BN=256 epilogue unchanged.
//   full[s]    leader's barrier: leader's producer arms 64 KB, both CTAs' TMA (.cta_group::2) complete_tx on it
//   empty[s]   per CTA, armed by the leader's tcgen05.commit.cta_group::2 multicast (mask 0b11)
//   tfull[t]   per CTA, same multicast commit after the last K block;  tempty[t]: leader's, 2*EW remote arrivals
//   work items one scheduler (leader, warp 2) -> both CTAs' item rings (st.shared::cluster + remote arrive)
// =============================================================================================
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_cl(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cl(uint32_t bar, uint32_t parity, int* err, int tag) {
  if (mbar_try_cl(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_cl(bar, parity)) {
    if (clock64() - t0 > 8000000000LL) {
      if (err) atomicExch(err, tag);
      __trap();
    }
  }
}
__device__ __forceinline__ void st_cluster_u32(uint32_t cluster_addr, uint32_t v) {
  asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}
// TMA load whose completion is signalled on a barrier that may live in the peer CTA of the pair
__device__ __forceinline__ void tma_load_3d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void mma_tf32_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void mma_commit_2sm(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(mask)
               : "memory");
}

template <int D4>
struct Cfg2 {
  static constexpr int BN = 256;                        // z columns per tile pair (128 staged by each CTA)
  static constexpr int RS = 4 * D4 + 4;
  static constexpr int SLOTS = 2;                       // 512 TMEM columns / 256
  static constexpr int STAGE_BYTES = (BM + BN / 2) * 128;   // per CTA: A half + B half = 32 KB
  static constexpr int STAGES = 6;
  static constexpr int COL_BYTES = BN * RS * 4;
  static constexpr int NBARS = 2 * STAGES + 2 * SLOTS + 4 + 2 * SCHED;
  static constexpr int SMEM_BYTES = 1024 + STAGES * STAGE_BYTES + 2 * COL_BYTES + 8 * NBARS + 64;
};

// work item = (256-row x tile pair, 256-column z tile); p.gx x tile pairs sweep the z tiles together
__device__ __forceinline__ bool item_coords2(const Params& p, long long item, int& xt, int& zt) {
  const long long per_group = (long long)p.gx * p.nzt;
  const int xg = (int)(item / per_group);
  const int r = (int)(item % per_group);
  zt = r / p.gx;
  xt = xg * p.gx + r % p.gx;
  return xt < p.nxt;
}

template <int D4, int EW, bool REFINE, bool TARGET, class KC>   // TARGET: GoOSE target epilogue (column OR, p.hit_words); KC: covariance function
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128 + 32 * EW, 1)
k_fantasy_tc2(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const Params p) {
  using C = Cfg2<D4>;
  constexpr int BN = C::BN, RS = C::RS, SLOTS = C::SLOTS, STAGES = C::STAGES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t tiles = base;
  const uint32_t colbuf = base + STAGES * C::STAGE_BYTES;
  const float* colbuf_ptr = reinterpret_cast<const float*>(base_ptr + STAGES * C::STAGE_BYTES);
  const uint32_t bars = colbuf + 2 * C::COL_BYTES;
  uint8_t* tail = base_ptr + STAGES * C::STAGE_BYTES + 2 * C::COL_BYTES + 8 * C::NBARS;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(tail);
  volatile int* sched_items = reinterpret_cast<volatile int*>(tail + 16);
  auto bar_full = [&](int s) { return bars + 8 * s; };
  auto bar_empty = [&](int s) { return bars + 8 * (STAGES + s); };
  auto bar_tfull = [&](int s) { return bars + 8 * (2 * STAGES + s); };
  auto bar_tempty = [&](int s) { return bars + 8 * (2 * STAGES + SLOTS + s); };
  auto bar_cfull = [&](int b) { return bars + 8 * (2 * STAGES + 2 * SLOTS + b); };
  auto bar_cempty = [&](int b) { return bars + 8 * (2 * STAGES + 2 * SLOTS + 2 + b); };
  auto bar_sfull = [&](int s) { return bars + 8 * (2 * STAGES + 2 * SLOTS + 4 + s); };
  auto bar_sempty = [&](int s) { return bars + 8 * (2 * STAGES + 2 * SLOTS + 4 + SCHED + s); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_empty(s), 1); }
    for (int s = 0; s < SLOTS; ++s) { mbar_init(bar_tfull(s), 1); mbar_init(bar_tempty(s), 2 * EW); }
    for (int b = 0; b < 2; ++b) { mbar_init(bar_cfull(b), 1); mbar_init(bar_cempty(b), EW); }
    // consumers of a work item: leader = producer, MMA, column loader + EW epilogue warps; peer = the same minus MMA
    for (int s = 0; s < SCHED; ++s) { mbar_init(bar_sfull(s), 1); mbar_init(bar_sempty(s), 5 + 2 * EW); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
  }
  __syncthreads();
  cluster_sync_all();          // the peer's barriers are initialised before anything is signalled across the pair
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_holder;

  int ss = 0; uint32_t sph = 0;
  auto next_item = [&](bool warp_wide) -> int {
    mbar_wait_cl(bar_sfull(ss), sph, p.err, 7);
    const int item = sched_items[ss];
    if (warp_wide) __syncwarp();
    if (!warp_wide || lane == 0) mbar_arrive_cluster(mapa_u32(bar_sempty(ss), 0));
    if (++ss == SCHED) { ss = 0; sph ^= 1; }
    return item;
  };

  if (warp == 2) {
    // ================================ scheduler (leader CTA only) ================================
    if (lane == 0 && rank == 0) {
      int s2 = 0; uint32_t ph2 = 0;
      const uint32_t peer_items = mapa_u32(smem_u32(const_cast<int*>(sched_items)), 1);
      for (;;) {
        long long item = (long long)atomicAdd(p.sched_counter, 1u);
        int v = (item < p.n_items) ? (p.item_list ? (int)p.item_list[item] : (int)item) : -1;
        mbar_wait_cl(bar_sempty(s2), ph2 ^ 1, p.err, 8);
        sched_items[s2] = v;
        st_cluster_u32(peer_items + 4 * s2, (uint32_t)v);
        mbar_arrive(bar_sfull(s2));
        mbar_arrive_cluster(mapa_u32(bar_sfull(s2), 1));
        if (++s2 == SCHED) { s2 = 0; ph2 ^= 1; }
        if (v < 0) break;
      }
    }
  } else if (warp == 0) {
    // ================================ TMA producer (both CTAs: own halves) ================================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (;;) {
        const int item = next_item(false);
        if (item < 0) break;
        int xt, zt;
        if (!item_coords2(p, item, xt, zt)) continue;
        for (int c = 0; c < p.nc; ++c)
          for (int kb = 0; kb < p.kblocks; ++kb) {
            mbar_wait_cl(bar_empty(stage), phase ^ 1, p.err, 1);
            if (rank == 0) mbar_expect_tx(bar_full(stage), 2 * C::STAGE_BYTES);
            const uint32_t full_leader = mapa_u32(bar_full(stage), 0);
            const uint32_t sa = tiles + stage * C::STAGE_BYTES;
            const int seg = p.split ? kb / p.nkb : 2, kk = (kb - (p.split ? seg : 0) * p.nkb) * BK;   // cross terms first (see above)
            tma_load_3d_2sm(sa, &tmA, full_leader, kk + (seg == 1 ? p.npad : 0), xt * 2 * BM + (int)rank * BM, c);
            tma_load_3d_2sm(sa + BM * 128, &tmB, full_leader, kk + (seg == 0 ? p.npad : 0), zt * BN + (int)rank * (BN / 2), c);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer (leader CTA only) ================================
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);
      int stage = 0; uint32_t phase = 0;
      int slot = 0; uint32_t sphase = 0;
      for (;;) {
        const int item = next_item(false);
        if (item < 0) break;
        int xt, zt;
        if (!item_coords2(p, item, xt, zt)) continue;
        for (int c = 0; c < p.nc; ++c) {
          mbar_wait_cl(bar_tempty(slot), sphase ^ 1, p.err, 2);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t tmem_d = tmem_base + (uint32_t)(slot * BN);
          for (int kb = 0; kb < p.kblocks; ++kb) {
            mbar_wait_cl(bar_full(stage), phase, p.err, 3);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t sa = tiles + stage * C::STAGE_BYTES;
            const uint64_t adesc = make_desc(sa), bdesc = make_desc(sa + BM * 128);
#pragma unroll
            for (int k = 0; k < BK / UK; ++k)
              mma_tf32_2sm(tmem_d, adesc + (uint64_t)(k * UK * 4 / 16), bdesc + (uint64_t)(k * UK * 4 / 16), idesc,
                           (kb | k) ? 1u : 0u);
            mma_commit_2sm(bar_empty(stage), 3);                          // frees the stage in BOTH CTAs
            if (kb == p.kblocks - 1) mma_commit_2sm(bar_tfull(slot), 3);    // accumulator complete in both TMEMs
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          if (++slot == SLOTS) { slot = 0; sphase ^= 1; }
        }
      }
    }
  } else if (warp == 3) {
    // ================================ column-record loader (both CTAs, all 256 columns) ================================
    if (lane == 0) {
      int b = 0; uint32_t bphase = 0;
      for (;;) {
        const int item = next_item(false);
        if (item < 0) break;
        int xt, zt;
        if (!item_coords2(p, item, xt, zt)) continue;
        for (int c = 0; c < p.nc; ++c) {
          mbar_wait(bar_cempty(b), bphase ^ 1, p.err, 4);
          mbar_expect_tx(bar_cfull(b), C::COL_BYTES);
          bulk_load_1d(colbuf + b * C::COL_BYTES, p.colrec + ((size_t)c * p.nzp + (size_t)zt * BN) * RS, C::COL_BYTES,
                       bar_cfull(b));
          if (++b == 2) { b = 0; bphase ^= 1; }
        }
      }
    }
  } else {
    // ================================ epilogue (warps 4 .. 4+EW-1), rows of THIS CTA's 128 candidates ================================
    const int q = warp & 3;
    const int half = (warp - 4) >> 2;
    constexpr int NCH = BN / 32 / (EW / 4);
    const int row = q * 32 + lane;
    int slot = 0; uint32_t sphase = 0;
    int b = 0; uint32_t bphase = 0;
    for (;;) {
      const int item = next_item(true);
      if (item < 0) break;
      int xt, zt;
      if (!item_coords2(p, item, xt, zt)) continue;
      const long long xrow = (long long)xt * 2 * BM + (long long)rank * BM + row;
      uint32_t bits[NCH];              // REFINE: safe at lo/mid/hi for every constraint so far
      uint32_t ubits[NCH];             // REFINE: unsafe at lo and hi for some constraint
#pragma unroll
      for (int h = 0; h < NCH; ++h) { bits[h] = 0xffffffffu; ubits[h] = 0u; }
      const uint64_t e_abs2 = pk2(p.e_abs, p.e_abs), d_mu2 = pk2(p.d_mu, p.d_mu), d_t2 = pk2(p.d_t, p.d_t);
      const KC kc(p.kernel);
      for (int c = 0; c < p.nc; ++c) {
        RowConsts<D4> rc;
        rc.load(p.rowrec + ((size_t)c * p.nxp + xrow) * RS);
        if (!KC::kIsSE) rc.kf = pk2(p.ksf2[c], p.ksf2[c]);
        mbar_wait(bar_cfull(b), bphase, p.err, 5);
        mbar_wait_cl(bar_tfull(slot), sphase, p.err, 6);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // pair-interleaved column records: RS packed pairs per two columns
        const uint64_t* cb = reinterpret_cast<const uint64_t*>(colbuf_ptr + (size_t)b * BN * RS) + (size_t)half * NCH * 16 * RS;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(slot * BN + half * NCH * 32);
#pragma unroll
        for (int h = 0; h < NCH; ++h) {
          uint32_t r[32];
          tmem_ld32(taddr + h * 32, r);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (REFINE) {
            uint32_t S, U;
            epilogue_chunk_refine<D4>(r, cb + (size_t)h * 16 * RS, rc, kc, e_abs2, d_mu2, d_t2, S, U);
            bits[h] &= S; ubits[h] |= U;
          } else {
            bits[h] &= epilogue_chunk<D4>(r, cb + (size_t)h * 16 * RS, rc, kc);
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) { mbar_arrive_cluster(mapa_u32(bar_tempty(slot), 0)); mbar_arrive(bar_cempty(b)); }
        if (++slot == SLOTS) { slot = 0; sphase ^= 1; }
        if (++b == 2) { b = 0; bphase ^= 1; }
      }
      if (TARGET) {
        // GoOSE target: column OR over the warp's 32 candidate rows, one atomicOr per 32-column word.  Padded rows and
        // columns are zero operands and must never set a bit, so rows >= nx and columns >= nz are masked first.
        const bool row_ok = xrow < p.nx;
#pragma unroll
        for (int h = 0; h < NCH; ++h) {
          const long long zc0 = (long long)zt * BN + (half * NCH + h) * 32;
          const uint32_t cm = zc0 + 32 <= p.nz ? 0xffffffffu : (zc0 >= p.nz ? 0u : (1u << (int)(p.nz - zc0)) - 1u);
          const uint32_t hw = __reduce_or_sync(0xffffffffu, row_ok ? bits[h] & cm : 0u);
          if (lane == 0 && hw) atomicOr(p.hit_words + (zc0 >> 5), hw);
          if (REFINE && p.amb_words) {
            const uint32_t amb = row_ok ? ~bits[h] & ~ubits[h] & cm : 0u;
            const uint32_t aw = __reduce_or_sync(0xffffffffu, amb);
            if (amb) atomicAdd(p.amb_count, (unsigned long long)__popc(amb));
            if (lane == 0 && aw) atomicOr(p.amb_words + (zc0 >> 5), aw);
          }
        }
      } else {
        int cnt = 0;
#pragma unroll
        for (int h = 0; h < NCH; ++h) cnt += __popc(bits[h]);
        if (xrow < p.nx && cnt) atomicAdd(p.counts + (p.row_perm ? p.row_perm[xrow] : xrow), cnt);
      }
      if (REFINE && xrow < p.nx && !(TARGET && p.amb_words)) {
#pragma unroll
        for (int h = 0; h < NCH; ++h) {
          uint32_t amb = ~bits[h] & ~ubits[h];              // neither settled safe nor settled unsafe
          if (amb) {
            const int n = __popc(amb);
            const unsigned long long base = atomicAdd(p.amb_count, (unsigned long long)n);
            if (p.amb_rows) { atomicAdd(p.amb_rows + (p.row_perm ? p.row_perm[xrow] : xrow), n); continue; }
            const int zc0 = zt * BN + (half * NCH + h) * 32;
            unsigned long long w = base;
            while (amb) {
              const int bpos = __ffs(amb) - 1; amb &= amb - 1;
              if ((long long)w < p.amb_cap) p.amb_list[w] = make_int2((int)xrow, zc0 + bpos);
              ++w;
            }
          }
        }
      }
    }
  }
  // ---- teardown: neither CTA may exit (or free TMEM) while the other can still signal it
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// FP32 record builders.  e = Cx - Bz + sum_k xx_k z_k = l - h s_c(z,x)  with  s_c = sum_k w_ck (z_k - x_k)^2:
//   SE:     h = log2(e)/2, l = log2 sf2_c, so that  k_c(z,x) = exp2(e)
//   MATERN: h = c (3 or 5), l = 0, so that  e = -c s = -t^2  (sf2_c is the per-constraint constant Params::ksf2)
//   row (candidate x):  xx_k = 2 h w_ck x_k ; Cx = l - h sum_k w_ck x_k^2 ; a = beta*sigma/(sigma^2+sn2) ;
//                       b' = beta^2/(sigma^2+sn2)
//   col (unsafe z):     z_k ; -Bz, Bz = h sum_k w_ck z_k^2 ; m_z = mean/Ystd ; s'_z = beta^2 var/Ystd^2
//                       (stored pair-interleaved: two adjacent columns form packed f32x2 operands)
// ---------------------------------------------------------------------------------------------
template <int D4, class KC>
__global__ void __launch_bounds__(256)
k_tc_records(FantasyConsts fc, long long n, long long npadrows, int is_row, const double* __restrict__ coords,
             const double* __restrict__ a, const double* __restrict__ b, float* __restrict__ rec, double esc,
             unsigned long long* __restrict__ stats) {
  constexpr int RS = 4 * D4 + 4;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int c = blockIdx.y;
  if (t >= npadrows) return;
  // rows: RS floats per candidate.  columns: pair-interleaved, entry k of column t at pair(t/2)*2*RS + 2*k + (t&1),
  // so that the epilogue reads (column 2p, column 2p+1) as one packed f32x2 operand
  float* o = is_row ? rec + ((size_t)c * npadrows + t) * RS : rec + ((size_t)c * npadrows + (t & ~1LL)) * RS + (t & 1);
  const int st = is_row ? 1 : 2;
  if (t >= n) {
    for (int k = 0; k < RS; ++k) o[k * st] = 0.f;
    if (!is_row) o[(4 * D4 + 1) * st] = -1e30f;         // padded z columns can never become safe
    return;
  }
  const double h = KC::kIsSE ? 0.5 * 1.4426950408889634 : MATERN(fc.kernel).c;
  double q = 0.0;
  for (int k = 0; k < 4 * D4; ++k) {
    const double x = (k < fc.d) ? coords[(size_t)k * n + t] : 0.0;
    const double w = (k < fc.d) ? fc.inv_ell[c][k] : 0.0;
    q += w * x * x;
    o[k * st] = is_row ? (float)(2.0 * h * w * x) : (float)x;
  }
  const double av = a[(size_t)c * n + t], bv = b[(size_t)c * n + t];
  if (stats) {   // maxima the host turns into the absolute error terms of the refining epilogue (non-negative doubles order like
                 // integers); reduced over the active lanes of the warp first: one atomic per warp and statistic
    const unsigned act = __activemask();
    unsigned long long m0 = (unsigned long long)__double_as_longlong(q);                           // sum_k w_k x_k^2
    unsigned long long m1 = is_row ? 0ULL : (unsigned long long)__double_as_longlong(fabs(av));     // |m_z|
    unsigned long long m2 = is_row ? 0ULL : (unsigned long long)__double_as_longlong(fmax(bv, 0.0));   // sigma_z^2
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long a0 = __shfl_xor_sync(act, m0, o), a1 = __shfl_xor_sync(act, m1, o), a2 = __shfl_xor_sync(act, m2, o);
      if ((act >> ((threadIdx.x & 31) ^ o)) & 1u) { m0 = max(m0, a0); m1 = max(m1, a1); m2 = max(m2, a2); }
    }
    if ((threadIdx.x & 31) == (unsigned)(__ffs(act) - 1)) {
      atomicMax(stats + (is_row ? 0 : 1), m0);
      if (!is_row) { atomicMax(stats + 2, m1); atomicMax(stats + 3, m2); }
    }
  }
  if (is_row) {
    o[4 * D4] = (float)((KC::kIsSE ? log2(fc.sf2[c]) : 0.0) - h * q);
    o[4 * D4 + 1] = (float)av;
    o[4 * D4 + 2] = (float)(fc.beta * fc.beta * bv);
  } else {
    o[(4 * D4) * st] = -(float)(h * q);                  // stored negated: e = (Cx + (-Bz)) + ...
    o[(4 * D4 + 1) * st] = (float)av;
    o[(4 * D4 + 2) * st] = (float)(fc.beta * fc.beta * bv);
  }
  // refinement band: sqrt(c1)*|v|, |v|^2 = sf2 - sigma^2 (rows: sigma^2 = 1/b - sn2; columns: b holds sigma^2); rounded UP
  const double s2 = is_row ? (1.0 / bv - fc.sn2[c]) : bv;
  o[(4 * D4 + 3) * st] = esc > 0.0 ? __double2float_ru(esc * sqrt(fmax(fc.sf2[c] - s2, 0.0))) : 0.f;
}

static int make_map(sbo_ctx* ctx, CUtensorMap* map, const float* base, int rowlen, long long rows, int nc, int box_rows) {
  cuuint64_t gdim[3] = {(cuuint64_t)rowlen, (cuuint64_t)rows, (cuuint64_t)nc};
  cuuint64_t gstr[2] = {(cuuint64_t)rowlen * 4, (cuuint64_t)rows * rowlen * 4};
  cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  // the driver entry point is resolved at run time so that the library has no link-time dependency on libcuda
  // (it must load, for symbol checks, on a machine without a GPU driver)
  typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static encode_fn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn)
      return sbo_fail(ctx, SBO_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    encode = (encode_fn)fn;
  }
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)base, gdim, gstr, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return sbo_fail(ctx, SBO_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
  return SBO_OK;
}

// the attribute is per device and cheap: set before every launch (a process may hold contexts on several GPUs)
template <int BN, int D4, int EW>
static int launch(sbo_ctx* ctx, const CUtensorMap& tmA, const CUtensorMap& tmB, const Params& p, int sms) {
  using C = Cfg<BN, D4>;
  SBO_CUDA(cudaFuncSetAttribute(k_fantasy_tc<BN, D4, EW>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
  const int grid = (int)((p.n_items < sms) ? p.n_items : sms);
  k_fantasy_tc<BN, D4, EW><<<grid, 128 + 32 * EW, C::SMEM_BYTES, ctx->stream>>>(tmA, tmB, p);
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

template <int D4, int EW, bool REFINE, bool TARGET, class KC>
static int launch2(sbo_ctx* ctx, const CUtensorMap& tmA, const CUtensorMap& tmB, const Params& p, int sms) {
  using C = Cfg2<D4>;
  const int clusters = sms / 2;
  SBO_CUDA((cudaFuncSetAttribute(k_fantasy_tc2<D4, EW, REFINE, TARGET, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES)));
  const int grid = 2 * (int)((p.n_items < clusters) ? p.n_items : clusters);
  k_fantasy_tc2<D4, EW, REFINE, TARGET, KC><<<grid, 128 + 32 * EW, C::SMEM_BYTES, ctx->stream>>>(tmA, tmB, p);
  SBO_LAUNCH_CHECK();
  return SBO_OK;
}

}  // namespace tc

// keys of the exact pruning (pairs.cu): sorted key_x[nx] (max side), key_z[nz] (min side), slot -> counts row;
// hit_words != null: GoOSE target (column OR into hit_words over the z slots; bounds mode: amb_words instead of amb_rows)
struct FantasyPruneArgs { const double* key_x; const double* key_z; const int* row_perm; long long* items_run;
                          int refine; int2* amb_list; unsigned long long* amb_count; long long amb_cap; int* amb_rows;
                          uint32_t* hit_words; uint32_t* amb_words; };
// per tile of `tile` consecutive sorted entries: max (x side) or min (z side) of the keys
__global__ void __launch_bounds__(256)
k_tile_keys(long long n, int tile, int want_max, const double* __restrict__ key, double* __restrict__ out) {
  __shared__ double red[8];
  const long long t0 = (long long)blockIdx.x * tile;
  double v = want_max ? -INFINITY : INFINITY;
  for (long long t = t0 + threadIdx.x; t < t0 + tile && t < n; t += 256) v = want_max ? fmax(v, key[t]) : fmin(v, key[t]);
  for (int o = 16; o > 0; o >>= 1) { const double w = __shfl_xor_sync(0xffffffffu, v, o); v = want_max ? fmax(v, w) : fmin(v, w); }
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) v = want_max ? fmax(v, red[w]) : fmin(v, red[w]);
    out[blockIdx.x] = v;
  }
}
// feasibility bitmask over the raster-ordered work items of the tcgen05 kernels (item -> (xt, zt) as item_coords*)
__global__ void __launch_bounds__(256)
k_item_mask(long long n_items, int gx, int nxt, int nzt, const double* __restrict__ qmax, const double* __restrict__ rmin,
            uint32_t* __restrict__ words) {
  const long long item = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool ok = false;
  if (item < n_items) {
    const long long per_group = (long long)gx * nzt;
    const int xg = (int)(item / per_group), r = (int)(item % per_group);
    const int zt = r / gx, xt = xg * gx + r % gx;
    ok = xt < nxt && rmin[zt] <= qmax[xt];
  }
  const uint32_t w = __ballot_sync(0xffffffffu, ok);
  if ((threadIdx.x & 31) == 0 && item < n_items) words[item >> 5] = w;
}


// exact pruning: raster-ordered list of the (x tile, z tile) pairs with min key_z <= max key_x (see pairs.cu k_key_z);
// item -> (xt, zt):  xg = item / (gx*nzt), r = item % (gx*nzt), zt = r / gx, xt = xg*gx + r % gx
int fantasy_build_items(sbo_ctx* ctx, long long nx, long long nz, int tile_x, int tile_z, int gx, const double* key_x,
                        const double* key_z, const long long** item_list, long long* n_list) {
  const int nxt = (int)cdiv(nx, tile_x), nzt = (int)cdiv(nz, tile_z);
  const long long n_raster = cdiv(nxt, gx) * gx * (long long)nzt;
  SBO_TRY(sbo_ensure(ctx, ctx->tile_keys, sizeof(double) * (size_t)(nxt + nzt)));
  double* qmax = (double*)ctx->tile_keys.p; double* rmin = qmax + nxt;
  k_tile_keys<<<nxt, 256, 0, ctx->stream>>>(nx, tile_x, 1, key_x, qmax);
  SBO_LAUNCH_CHECK();
  k_tile_keys<<<nzt, 256, 0, ctx->stream>>>(nz, tile_z, 0, key_z, rmin);
  SBO_LAUNCH_CHECK();
  SBO_TRY(sbo_ensure(ctx, ctx->item_mask, sizeof(uint32_t) * (size_t)cdiv(n_raster, 32)));
  k_item_mask<<<(unsigned)cdiv(n_raster, 256), 256, 0, ctx->stream>>>(n_raster, gx, nxt, nzt, qmax, rmin, (uint32_t*)ctx->item_mask.p);
  SBO_LAUNCH_CHECK();
  SBO_TRY(compact_mask(ctx, (const uint32_t*)ctx->item_mask.p, n_raster, ctx->item_list, n_list));
  *item_list = (const long long*)ctx->item_list.p;
  return SBO_OK;
}

int fantasy_tc_run(sbo_ctx* ctx, const FantasyConsts& fc, int split, long long nx, long long nz, long long nxp,
                   long long nzp, const float* Vx, const float* Vz, const double* aux_x, const double* aux_z, int* counts_c,
                   const FantasyPruneArgs* pr) {
  const int d = fc.d, nc = fc.nc;
  const int D4 = d <= 4 ? 1 : 2;
  const int RS = 4 * D4 + 4;
  SBO_REQUIRE(fc.npad % tc::BK == 0, "npad must be a multiple of 32");
  SBO_REQUIRE(nxp % 256 == 0 && nzp % 256 == 0, "padded row counts must be multiples of 256");
  SBO_TRY(sbo_ensure(ctx, ctx->tc_row, sizeof(float) * (size_t)nc * nxp * RS));
  SBO_TRY(sbo_ensure(ctx, ctx->tc_col, sizeof(float) * (size_t)nc * nzp * RS));
  SBO_TRY(sbo_ensure(ctx, ctx->tc_err, 2 * sizeof(int)));            // [0] error tag, [1] work-item counter
  SBO_CUDA(cudaMemsetAsync(ctx->tc_err.p, 0, 2 * sizeof(int), ctx->stream));
  const double* xn = aux_x; const double* ax = xn + (size_t)d * nx; const double* bx = ax + (size_t)nc * nx;
  const double* zn = aux_z; const double* mz = zn + (size_t)d * nz; const double* sz = mz + (size_t)nc * nz;
  float* rowrec = (float*)ctx->tc_row.p;
  float* colrec = (float*)ctx->tc_col.p;
  // refinement band of the split mode: c1 = 2^-20 (operand split: representation + dropped lo.lo) + one ulp (2^-23) of the
  // running sum per tensor-core accumulation step of the hi.hi segment (K/8 steps); the cross segments are accumulated
  // first at 2^-11 of that size.  e_abs / d_mu / d_t: ex2.approx, FP32 records and the FP32 epilogue arithmetic.
  // Single-pass TF32 (option fantasy_refine = 2): the operand rounding itself, 2^-11 per operand -> 2^-10 (+2^-22) per product.
  const bool refine = pr && pr->refine;
  const double c1 = refine ? ((split ? 9.5367431640625e-07 : 9.7680091857910156e-04) + (fc.npad / 8) * 1.1920928955078125e-07) : 0.0;
  const double esc = refine ? sqrt(c1) : 0.0;
  tc::Params p{};
  const bool target = pr && pr->hit_words;
  p.hit_words = target ? pr->hit_words : nullptr;
  unsigned long long* stats = nullptr;
  if (refine) {
    p.amb_list = pr->amb_list; p.amb_count = pr->amb_count; p.amb_cap = pr->amb_cap; p.amb_rows = pr->amb_rows; p.amb_words = pr->amb_words;
    SBO_TRY(sbo_ensure(ctx, ctx->tc_stats, 4 * sizeof(unsigned long long)));
    stats = (unsigned long long*)ctx->tc_stats.p;
    SBO_CUDA(cudaMemsetAsync(stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
  }
  ev_begin(ctx, 6);
  const bool se = fc.kernel == SBO_KERNEL_SE;
  SBO_TRY((with_int<1, 2>(D4, [&](auto d4) { return with_kernel(fc.kernel, [&](auto kc) -> int {
    tc::k_tc_records<d4, decltype(kc)><<<dim3((unsigned)cdiv(nxp, 256), nc), 256, 0, ctx->stream>>>(fc, nx, nxp, 1, xn, ax, bx, rowrec, esc, stats);
    SBO_LAUNCH_CHECK();
    tc::k_tc_records<d4, decltype(kc)><<<dim3((unsigned)cdiv(nzp, 256), nc), 256, 0, ctx->stream>>>(fc, nz, nzp, 0, zn, mz, sz, colrec, esc, stats);
    SBO_LAUNCH_CHECK();
    return SBO_OK;
  }); })));
  if (refine) {
    // absolute error terms of the FP32 epilogue from the data (one small read-back):
    //   exponent  e = (Cx - Bz) + sum xx_k z_k : 12*D4+3 roundings (inputs and FMAs) of magnitudes <= T = |log2 sf2| + 2h(Ax + Az),
    //             k = ex2.approx(e) (2 ulp), cov = k - acc (1 rounding of <= 2 sf2)             -> e_abs
    //   mean      mu' = cov*a + m : two roundings of <= |m|max + beta*sqrt(sf2) (a*|cov| <= beta*sigma_z)   -> d_mu
    //   variance  t = s' - cov^2 b', compared with mu'^2 near mu'^2 ~ t <= beta^2 (s_z + sf2)     -> d_t
    // Matern (records scaled by c, e = -c s <= 0, k = sf2 P(t) exp(-t) with t = sqrt(max(-e, 0))):
    //   exponent  the same 12*D4+3 roundings, of magnitudes <= T = c (Ax + Az) (no log2 sf2 term).  |dk/de| = |dk/ds| / c
    //             <= kappa sf2 / 2 with kappa = max_t ((1-2q) + q t) e^-t = 1 (3/2) or 1/3 (5/2), and the clamp at 0 only
    //             moves e towards the true value: error in k <= kappa/2 sf2 u (12*D4+3) T
    //   value     with t = sqrt(-e) exact, the FP32 evaluation adds at most 17.3 u sf2, taken as 32 u sf2: sqrt.approx
    //             (<= 8 u relative in t; t |dk/dt| = sf2 t^2 ((1-2q) + q t) e^-t <= 0.61 sf2 -> 4.9 u), the argument -t log2(e)
    //             (2 u relative -> ln2 * 2u t log2(e) relative in k; t P(t) e^-t <= 1.2 -> 2.4 u), ex2.approx (4 u),
    //             the polynomial (3 u), the two products (2 u) and sf2 in FP32 (1 u): every t^j e^-t is bounded
    //   cov = k - acc: one rounding of <= 2 sf2                                                   -> e_abs
    double st[4];
    SBO_CUDA(cudaMemcpyAsync(st, stats, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    SBO_CUDA(cudaStreamSynchronize(ctx->stream));
    double sf2max = 0.0, lsf = 0.0;
    for (int c = 0; c < nc; ++c) { sf2max = fmax(sf2max, fc.sf2[c]); lsf = fmax(lsf, fabs(log2(fc.sf2[c]))); }
    const double h = 0.5 * 1.4426950408889634, u = 5.9604644775390625e-08;           // u = 2^-24
    if (se) {
      const double T = lsf + 2.0 * h * (st[0] + st[1]);
      p.e_abs = (float)(sf2max * (0.6931471805599453 * u * (12 * D4 + 3) * T * 1.05 + 8.0 * u) + 4.0 * u * sf2max);
    } else {
      const MATERN mk(fc.kernel);
      const double kappa = mk.q > 0.0 ? 1.0 / 3.0 : 1.0;
      const double T = mk.c * (st[0] + st[1]);
      p.e_abs = (float)(sf2max * (0.5 * kappa * u * (12 * D4 + 3) * T * 1.05 + 32.0 * u) + 4.0 * u * sf2max);
    }
    p.d_mu = (float)(4.0 * u * (st[2] + fc.beta * sqrt(sf2max)) + 1e-9);
    p.d_t = (float)(8.0 * u * fc.beta * fc.beta * (st[3] + sf2max) + 1e-9);
  }
  int* err = (int*)ctx->tc_err.p;
  // variant: bit 0: BN = 256, bit 1: 8 epilogue warps, bit 2: 2-CTA pairs (cta_group::2, 256 x 256 tile pairs);
  // < 0 = auto: 2-CTA pairs (a third less L2->SM operand traffic, 6 stages); 8 epilogue warps when the epilogue
  // outweighs the MMAs (short K) or carries 12-float records (d > 4)
  int variant = (int)ctx->opt_fantasy_variant;
  if (variant < 0) variant = 5 | ((fc.npad <= 256 || D4 == 2) ? 2 : 0);
  if (refine) variant |= 7;        // the refining epilogue exists in the 2-CTA kernel only; it is heavier: 8 epilogue warps
  if (target) variant |= 4;        // so does the column-OR epilogue of the GoOSE target
  if (!se) variant |= 4;           // and the Matern epilogue
  // tile geometry of the chosen kernel and the raster of its work items
  const bool two = (variant & 4) != 0;
  const int tile_x = two ? 2 * tc::BM : tc::BM, tile_z = (two || (variant & 1)) ? 256 : 128;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  const int gx = two ? (ctx->opt_fantasy_gx > 0 ? (int)ctx->opt_fantasy_gx : (sms / 2 + 3) / 4) : tc::GX;
  const int nxt = (int)cdiv(nx, tile_x), nzt = (int)cdiv(nz, tile_z);
  const long long n_raster = cdiv(nxt, gx) * gx * (long long)nzt;
  SBO_REQUIRE(n_raster < 2000000000LL, "too many tile pairs for one launch");
  const long long* item_list = nullptr;
  long long n_list = n_raster;
  const int* row_perm = pr ? pr->row_perm : nullptr;
  if (pr && pr->key_x && pr->key_z)
    SBO_TRY(fantasy_build_items(ctx, nx, nz, tile_x, tile_z, gx, pr->key_x, pr->key_z, &item_list, &n_list));
  if (pr && pr->items_run) *pr->items_run = n_list * (long long)tile_x * tile_z;   // pairs per constraint actually evaluated
  ev_end(ctx);            // record prep = phase 6
  ev_begin(ctx, 4);       // the GEMM kernel alone = phase 4 (closed by the caller)
  // the TMA maps and the work of both kernels; a 2-CTA pair stages half of its z tile in each CTA
  CUtensorMap tmA, tmB;
  const int rowlen = split ? 2 * fc.npad : fc.npad;
  SBO_TRY(tc::make_map(ctx, &tmA, Vx, rowlen, nxp, nc, tc::BM));
  SBO_TRY(tc::make_map(ctx, &tmB, Vz, rowlen, nzp, nc, two ? tile_z / 2 : tile_z));
  p.nc = nc; p.nkb = fc.npad / tc::BK; p.kblocks = split ? 3 * p.nkb : p.nkb; p.npad = fc.npad; p.split = split;
  p.nx = nx; p.nz = nz; p.nxp = nxp; p.nzp = nzp;
  p.nxt = nxt; p.nzt = nzt; p.gx = gx; p.n_items = n_list;
  p.rowrec = rowrec; p.colrec = colrec; p.counts = counts_c; p.err = err;
  p.sched_counter = (unsigned int*)(err + 1);
  p.item_list = item_list; p.row_perm = row_perm;
  p.kernel = fc.kernel;
  for (int c = 0; c < nc; ++c) p.ksf2[c] = (float)fc.sf2[c];
  if (p.n_items == 0) return SBO_OK;
  return with_int<1, 2>(D4, [&](auto d4) { return with_flag(variant & 2, [&](auto ew8) {
    if (two)            // 2-CTA pairs (cta_group::2), BN = 256
      return with_flag(refine, [&](auto r) { return with_flag(target, [&](auto t) { return with_kernel(fc.kernel, [&](auto kc) {
        return tc::launch2<d4, (ew8 ? 8 : 4), r, t, decltype(kc)>(ctx, tmA, tmB, p, sms);
      }); }); });
    return with_flag(variant & 1, [&](auto bn256) { return tc::launch<(bn256 ? 256 : 128), d4, (ew8 ? 8 : 4)>(ctx, tmA, tmB, p, sms); });
  }); });
}
