// K1 + K2, fast mode, "f8c" operand format: one fp16 product plus two e4m3 correction products on a CTA pair.
// Same contract as k_posterior_fast (posterior_fast.cu): mu and var per candidate of one GP, tolerance rtol 1e-3.
//
//   V = K* . (s sigma_f2 L^-1)^T,  A = K* = k'(r) in (0,1] generated on chip,  B = s sigma_f2 L^-1 (planes from K3)
//   A = A_h + A_l   (A_h = fp16(A), exact residual A_l, |A_l| <= 2^-12)
//   B = B_h + B_l   (B_h = fp16(B), exact residual B_l, |B_l| <= 4 with max |B| scaled into [8192, 16384))
//   V ~= A_h B_h^T                              kind::f16      (K = 16 per instruction)         1   tensor unit
//      + e4m3(2^12 A_l) . e4m3(2^-12 B)^T       kind::f8f6f4   (K = 32: twice the MAC rate)     1/2
//      + e4m3(A) . e4m3(B_l)^T                  kind::f8f6f4                                    1/2
// All three accumulate into the same FP32 TMEM tile (every scale is a power of two, so the three products carry
// the same factor s).  The correction operands only need the ~2^-5 relative precision e4m3 has: they multiply
// residuals that are already 2^-12 of the operands.  2.0 tensor units per algorithmic MAC instead of the 3.0 of the
// 16-bit x3 split; measured sigma error against FP64 in DESIGN.md section 4 (the refresh selects this format only
// while the conditioning proxy of the factor stays below the measured limit).
//
// One CTA PAIR (cluster of 2, tcgen05 cta_group::2) owns 256 candidates: UMMA M = 256 (128 rows per CTA),
// N <= 256, each CTA TMA-loads only ITS half of every B tile, which halves the B traffic through shared memory
// and L2 per candidate -- the two limits the single-CTA kernel runs into (DESIGN.md section 4).
//   warp 0        B producer (both CTAs): this CTA's rows of the unit's three planes, bytes counted on the leader
//   warp 1        MMA issuer (leader CTA): per (256-column chunk, 64-deep K-block) 4 x f16 + 2 x 2 x f8f6f4
//   warp 2        TMEM allocator (512 columns = two 256-column accumulator chunks per CTA), then the candidate
//                 coordinates of the next tile (counter generator / conversion, scaled and centred)
//   warp 3        one thread: train slices of the coming K-blocks by TMA bulk copies (ring of 4), copies of the
//                 generated K* stages to / from the per-CTA cache in L2
//   warps 4-7     epilogue: tcgen05.ld, square + row sum, var = sigma_f2 - sum V^2 / s^2
//   warps 8..     K1 generators (8 or 16 warps): distances in FP32 (packed FFMA2), Matern-5/2 / RBF via MUFU,
//                 fp16 / e4m3 planes written straight into the UMMA operand layouts (SWIZZLE_128B / SWIZZLE_64B);
//                 no barrier between generator warps inside a tile (mbarrier rings only)
// L^-1 is lower triangular: chunk c needs K-blocks kb <= 4c+3 only, and on the four diagonal K-blocks of a chunk
// the rows above the diagonal band are zero, so N shrinks to 192 / 128 / 64 -- in pair mode by letting each CTA
// fetch a different row range of the band (CTA r loads rows r0 + r N/2 .. of the chunk) and offsetting the
// accumulator columns by r0.
// TMEM holds two 256-column accumulators ("slots"); a tile with more chunks walks a STEP SCHEDULE built on the host
// (f8_build_schedule): every K-block is generated exactly once, in order, and multiplied into the chunks open at
// that moment; a chunk that opens later (when a slot has been drained) gets the blocks it missed streamed back from
// a per-CTA cache in L2, and those reload steps are placed where the tensor core would otherwise wait for the
// generators (K1 costs ~3 units of MMA time per block).  All roles walk the same schedule, one 32-bit word per step.
#include <cuda_fp8.h>

#include <deque>
#include <vector>

#include "umma.cuh"
#include "acq_math.cuh"
#include "gen8.cuh"

#define F8_HI_BYTES 16384   // 128 rows x 64 fp16 (SWIZZLE_128B)
#define F8_P8_BYTES 8192    // 128 rows x 64 e4m3 (SWIZZLE_64B)
#define F8_OFF_C1 F8_HI_BYTES                  // A: e4m3(2^12 A_l)   B: e4m3(2^-12 B)
#define F8_OFF_C2 (F8_HI_BYTES + F8_P8_BYTES)  // A: e4m3(A)          B: e4m3(B_l)

// UMMA shared-memory descriptor, K-major, SWIZZLE_64B: rows of 64 B, 8-row groups 512 B apart
__device__ __forceinline__ uint64_t make_sdesc64(uint32_t saddr) {
  const uint32_t lo = ((saddr & 0x3FFFF) >> 4) | (1u << 16);
  const uint32_t hi = 32u | (1u << 14) | (4u << 29);                   // SBO = 512 B, version 1, SWIZZLE_64B
  return ((uint64_t)hi << 32) | lo;
}
__device__ __forceinline__ void umma_f8_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}

#define F8_NSL 4            // train-slice ring depth
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void st_release_shared(uint32_t a, uint32_t v) {
  asm volatile("st.release.cta.shared::cta.u32 [%0], %1;\n" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_shared(uint32_t a) {
  uint32_t v;
  asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];\n" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts64(uint32_t a, uint32_t x, uint32_t y) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};\n" ::"r"(a), "r"(x), "r"(y) : "memory");
}
// the same with a compile-time byte offset folded into the instruction (no address arithmetic per store)
template <int OFF>
__device__ __forceinline__ void sts128_at(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0+%5], {%1, %2, %3, %4};\n" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w), "n"(OFF) : "memory");
}
template <int OFF>
__device__ __forceinline__ void sts64_at(uint32_t a, uint32_t x, uint32_t y) {
  asm volatile("st.shared.v2.b32 [%0+%3], {%1, %2};\n" ::"r"(a), "r"(x), "r"(y), "n"(OFF) : "memory");
}

#define F8_TRACE_N 8192
#ifndef F8_TRACING
#define F8_TRACING 0      // build with EXTRA=-DF8_TRACING=1 and run with OMBO_FAST_PROFILE=2 (scripts/trace_fast8.py)
#endif
// event trace (timing experiments): CTA 0 only, tiles 2 and 3, one region per role
#if !F8_TRACING
#define F8_TRACE(role, code) do { } while (0)
#define F8_TRACE_G(code) do { } while (0)
#define F8_TRACE_E(code) do { } while (0)
#else
#define F8_TRACE_G(code) do { if (trole >= 0) F8_TRACE(trole, code); } while (0)
#define F8_TRACE_E(code) do { if (warp == 4 && lane == 0) F8_TRACE(4, code); } while (0)
#define F8_TRACE(role, code)                                                                   \
  do {                                                                                         \
    if (tron && it >= 2 && it < 4 && tr_n[role] < F8_TRACE_N)                                  \
      prm.trace[(role) * F8_TRACE_N + tr_n[role]++] = (clock64() << 8) | (long long)(code);    \
  } while (0)
#endif

// schedule word: one step = one K-block (fresh: generated now / cached: reloaded) multiplied into <= 2 chunks
#define SW_KB(w) ((int)((w) & 0xFFu))
#define SW_FRESH(w) (((w) >> 8) & 1u)
#define SW_STORE(w) (((w) >> 9) & 1u)                            // fresh block that a later chunk reloads
#define SW_CHUNK(w, slot) ((int)(((w) >> (10 + 6 * (slot))) & 63u) - 1)   // chunk in TMEM slot 0 / 1, -1 = none
#define SW_FIRST(w, slot) (((w) >> (22 + (slot))) & 1u)          // first block of that chunk (accumulator reset)
#define SW_DONE(w, slot) (((w) >> (24 + (slot))) & 1u)           // last block of that chunk (epilogue may drain)
#define SW_MEAN(w) (((w) >> 26) & 1u)                            // bound schedule: fresh block that feeds the mean only

struct F8Maps {            // tensor maps of the three B planes (128-row and 32-row boxes) and of the K* cache
  CUtensorMap hi128, hi32, c1_128, c1_32, c2_128, c2_32, kc;
};

// BOUND: the kernel walks a bound schedule (f8_build_schedule, bound_chunks > 0).  Its MEAN steps generate k' and the
// mean exactly as a full launch does and multiply nothing, so mu is the full launch's and var is the upper bound
// sigma_f2 - (the first chunks' sum of V^2) >= var.  A separate instantiation: the full kernel carries no mean-step code.
template <int DP, int R, int GW, bool MATERN, bool BOUND>
__global__ void __launch_bounds__((8 + GW) * 32, 1)
k_posterior_fast8(const __grid_constant__ F8Maps maps, const FastParams prm) {
  constexpr int NSTA = 3, NSTB = 3;
  constexpr int NSL = F8_NSL;                   // train-slice ring (TMA bulk copies, one slice per fresh K-block)
  constexpr int GEN_WARPS = GW;
  constexpr int CW = 256;
  constexpr int XT_STRIDE = (DP + 2) * FK;     // floats per slice: DP coordinate rows, sigma_f2 alpha, |b|^2
  constexpr uint32_t SLICE_BYTES = XT_STRIDE * 4;
  // D = f32, A = B = fp16 / e4m3 (format code 0 in both kinds), K-major, M = 256 (pair); N is patched per unit
  constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(256 >> 4) << 24);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int d = prm.gp.d, np = prm.gp.n_pad;
  const int nkb = np / FK;
  const long long n_tiles = (prm.m + FM - 1) / FM;
  const long long n_iter = (n_tiles + gridDim.x - 1) / gridDim.x;   // both CTAs of a pair walk the same sequence
  const uint32_t crank = cluster_rank();
  const bool leader = crank == 0;
  const int n_steps = prm.n_steps;
  // columns of chunk c that K-block kb touches: [r0, r0 + ncols) of the chunk (rows of L^-1 above the diagonal band
  // and beyond n_pad are zero)
  auto unit_r0 = [&](int c, int kb) { return max(0, kb - 4 * c) * 64; };
  auto unit_ncols = [&](int c, int kb) { return min(CW, np - c * CW) - unit_r0(c, kb); };

  unsigned char *sA = fast_smem + ((1024u - (smem_u32(fast_smem) & 1023u)) & 1023u);
  unsigned char *sB = sA + NSTA * STAGE_BYTES;
  float *xc = (float *)(sB + NSTB * STAGE_BYTES);              // [2][DP][128] scaled candidate coords (double buffered)
  float *xt = xc + 2 * (size_t)DP * FM;                        // [NSL][DP + 2][64] train slices
  float *mu_sm = xt + (size_t)NSL * XT_STRIDE;                 // [2][4][128] mean partials (double buffered by tile)
  uint64_t *bars = (uint64_t *)(((uintptr_t)(mu_sm + 8 * FM) + 15) & ~(uintptr_t)15);
  uint64_t *a_full = bars, *a_empty = bars + 3, *b_full = bars + 6, *b_empty = bars + 9;
  uint64_t *t_full = bars + 12, *t_empty = bars + 14;
  uint64_t *s_full = bars + 16, *s_empty = bars + 20;           // train-slice ring
  uint64_t *a_written = bars + 24;                              // "all local generator warps have written stage s"
  uint64_t *xc_full = bars + 27, *xc_empty = bars + 29;
  uint32_t *tmem_slot = (uint32_t *)(bars + 32);
  double *inv_ell = (double *)(bars + 34);
  uint32_t *store_seq = (uint32_t *)(bars + 50);               // [128] warp 3's private table (K* cache store order)
  uint32_t *landed = store_seq + 128;                          // (spare words)
  // the step schedule is staged in shared memory (every role reads a word per step, and with this much shared
  // memory carved out there is next to no L1 left for a global table); very long schedules stay in global memory
  uint64_t *mu_full = (uint64_t *)(landed + 4);                // [2] fused epilogue: the tile's mean partials are in mu_sm
  double *red_v = (double *)(mu_full + 2);                     // [4] + [4] per-warp arg-max of the fused epilogue
  long long *red_i = (long long *)(red_v + 4);
  uint32_t *sched_sm = (uint32_t *)(red_i + 4);
  const uint32_t *sched = prm.sched_in_smem ? (const uint32_t *)sched_sm : prm.sched;
  if (prm.sched_in_smem)
    for (int i = tid; i < n_steps; i += blockDim.x) sched_sm[i] = __ldg(prm.sched + i);
  // fused acquisition: stripe bounds of the 2-D EHVI as FP32, behind the schedule
  const bool fuse = prm.fuse.on != 0;
  float *ystr = (float *)(sched_sm + (prm.sched_in_smem ? n_steps : 0));
  if (fuse)
    for (int i = tid; i < 2 * (prm.fuse.n_pf + 2); i += blockDim.x) ystr[i] = (float)prm.fuse.stripes[i];

  if (tid == 0) {
    for (int j = 0; j < DP; ++j) inv_ell[j] = j < d ? 1.0 / prm.gp.ell[j] : 0.0;
    *landed = 0u;
    for (int s = 0; s < NSTA; ++s) {
      mbar_init(smem_u32(&a_full[s]), 2 * GEN_WARPS);
      mbar_init(smem_u32(&a_empty[s]), 2);                      // the MMA's commit + this CTA's cache thread
      mbar_init(smem_u32(&a_written[s]), GEN_WARPS);
    }
    for (int s = 0; s < NSTB; ++s) { mbar_init(smem_u32(&b_full[s]), 1); mbar_init(smem_u32(&b_empty[s]), 1); }
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&t_full[s]), 1); mbar_init(smem_u32(&t_empty[s]), 8);
      mbar_init(smem_u32(&xc_full[s]), 1); mbar_init(smem_u32(&xc_empty[s]), GEN_WARPS);
      mbar_init(smem_u32(&mu_full[s]), GEN_WARPS);
    }
    for (int s = 0; s < NSL; ++s) { mbar_init(smem_u32(&s_full[s]), 1); mbar_init(smem_u32(&s_empty[s]), GEN_WARPS); }
    fence_mbar_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n" ::);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                       // the peer arrives on / loads into this CTA's barriers and smem
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const bool pon = prm.prof != nullptr;
#if F8_TRACING
  const bool tron = prm.trace != nullptr && blockIdx.x == 0;
  int tr_n[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif
  // 24 warps leave 80 registers per thread, which the generator loop does not fit in (it spilled and re-derived
  // its addresses every K-block).  The four role warps and the epilogue give registers back, the generator
  // warpgroups take them: the pool is what the CTA was launched with, 768 x 80 = 128 x 56 + 128 x 72 + 512 x 88.
  // (the role code of a warpgroup has to sit behind ITS setmaxnreg for ptxas to allocate by the new limit)
  if (warp < 4) {
  if (GW == 16) asm volatile("setmaxnreg.dec.sync.aligned.u32 56;\n");
  if (warp == 0) {
    // =============================== B producer (both CTAs) ===============================
    if (elect_one() && !(prm.dbg & 128)) {
      uint32_t st = 0, ph = 0;
      long long w_bempty = 0; const long long t_start = clock64();
      for (long long it = 0; it < n_iter; ++it) {
        for (int si = 0; si < n_steps; ++si) {
          const uint32_t w = sched[si];
          const int kb = SW_KB(w);
          for (int slot = 0; slot < 2; ++slot) {
            const int c = SW_CHUNK(w, slot);
            if (c < 0) continue;
            const int ncols = unit_ncols(c, kb), rows = ncols >> 1;          // rows of the band this CTA holds
            const int row0 = c * CW + unit_r0(c, kb) + (int)crank * rows;
            mbar_wait_prof(smem_u32(&b_empty[st]), ph ^ 1, 64, w_bempty, pon);
            F8_TRACE(0, kb * 8 + c);
            const uint32_t dst = smem_u32(sB + st * STAGE_BYTES);
            // the leader alone arms its barrier, with the bytes of BOTH halves (256 B per band row over the planes)
            const uint32_t full = mapa_rank(smem_u32(&b_full[st]), 0);
            if (leader) mbar_expect_tx(smem_u32(&b_full[st]), (uint32_t)(ncols * 256));
            if (rows == 128) {
              tma_load_2d_2sm(dst, &maps.hi128, full, kb * FK, row0);
              tma_load_2d_2sm(dst + F8_OFF_C1, &maps.c1_128, full, kb * FK, row0);
              tma_load_2d_2sm(dst + F8_OFF_C2, &maps.c2_128, full, kb * FK, row0);
            } else {
              for (int rr = 0; rr < rows; rr += 32) {
                tma_load_2d_2sm(dst + (uint32_t)(rr * 128), &maps.hi32, full, kb * FK, row0 + rr);
                tma_load_2d_2sm(dst + F8_OFF_C1 + (uint32_t)(rr * 64), &maps.c1_32, full, kb * FK, row0 + rr);
                tma_load_2d_2sm(dst + F8_OFF_C2 + (uint32_t)(rr * 64), &maps.c2_32, full, kb * FK, row0 + rr);
              }
            }
            if (++st == NSTB) { st = 0; ph ^= 1; }
          }
        }
      }
      if (pon) { prm.prof[blockIdx.x * 16 + 0] = w_bempty; prm.prof[blockIdx.x * 16 + 1] = clock64() - t_start; }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer (leader CTA) ==============================
    if (leader && elect_one() && !(prm.dbg & 128)) {
      uint32_t sa = 0, pa = 0, sb = 0, pb = 0, tph = 0;
      long long w_afull = 0, w_bfull = 0, w_tempty = 0;
      for (long long it = 0; it < n_iter; ++it) {
        for (int si = 0; si < n_steps; ++si) {
          const uint32_t w = sched[si];
          const int kb = SW_KB(w);
          if (BOUND && SW_MEAN(w)) continue;                // nothing to multiply, no stage
          F8_TRACE(1, 0x80 | (kb & 31));
          mbar_wait_prof(smem_u32(&a_full[sa]), pa, MMA_SLEEP_NS, w_afull, pon);
          F8_TRACE(1, 0xC0 | (kb & 31));
          tc_fence_after();
          const uint32_t a_hi = smem_u32(sA + sa * STAGE_BYTES);
          for (int slot = 0; slot < 2; ++slot) {
            const int c = SW_CHUNK(w, slot);
            if (c < 0) continue;
            const uint32_t first = SW_FIRST(w, slot);
            if (first) {                                   // the slot's previous chunk must have been drained
              mbar_wait_prof(smem_u32(&t_empty[slot]), ((tph >> slot) & 1) ^ 1, MMA_SLEEP_NS, w_tempty, pon);
              tph ^= (1u << slot);
              tc_fence_after();
            }
            const int r0 = unit_r0(c, kb), ncols = unit_ncols(c, kb);
            const uint32_t dcol = tmem_base + (uint32_t)(slot * CW + r0);
            const uint32_t idesc = IDESC | ((uint32_t)(ncols >> 3) << 17);
            mbar_wait_prof(smem_u32(&b_full[sb]), pb, MMA_SLEEP_NS, w_bfull, pon);
            F8_TRACE(1, (kb & 15) * 4 + (c & 3));
            tc_fence_after();
            const uint32_t b_hi = smem_u32(sB + sb * STAGE_BYTES);
            if (!(prm.dbg & 1)) {
#pragma unroll
              for (int ks = 0; ks < FK / 16; ++ks)
                umma_bf16_2sm(dcol, make_sdesc(a_hi + ks * 32), make_sdesc(b_hi + ks * 32), idesc, (!first || ks > 0) ? 1u : 0u);
              if (!(prm.dbg & 4)) {
#pragma unroll
                for (int ks = 0; ks < FK / 32; ++ks)
                  umma_f8_2sm(dcol, make_sdesc64(a_hi + F8_OFF_C1 + ks * 32), make_sdesc64(b_hi + F8_OFF_C1 + ks * 32), idesc, 1u);
#pragma unroll
                for (int ks = 0; ks < FK / 32; ++ks)
                  umma_f8_2sm(dcol, make_sdesc64(a_hi + F8_OFF_C2 + ks * 32), make_sdesc64(b_hi + F8_OFF_C2 + ks * 32), idesc, 1u);
              }
            }
            umma_commit_2sm(smem_u32(&b_empty[sb]));
            if (SW_DONE(w, slot)) umma_commit_2sm(smem_u32(&t_full[slot]));      // chunk complete
            if (++sb == NSTB) { sb = 0; pb ^= 1; }
          }
          umma_commit_2sm(smem_u32(&a_empty[sa]));
          F8_TRACE(1, 0x40 | (kb & 31));
          if (++sa == NSTA) { sa = 0; pa ^= 1; }
        }
      }
      if (pon) { prm.prof[blockIdx.x * 16 + 2] = w_afull; prm.prof[blockIdx.x * 16 + 3] = w_bfull; prm.prof[blockIdx.x * 16 + 4] = w_tempty; }
    }
  } else if (warp == 2) {
    // =============================== candidate coordinates of the next tile ===============
    // -2 x the centred, length-scaled coordinates of tile `it` into xc[it & 1] while the generators work on tile
    // it - 1 (FP64 counter generator / conversion: ~20 k cycles per tile off the generators' critical path).
    // xc_full[b]: filled (one arrival by this warp), xc_empty[b]: every generator warp has its rows in registers.
    for (long long it = 0; it < n_iter; ++it) {
      const int b = (int)(it & 1);
      const uint32_t u = (uint32_t)(it >> 1);
      const long long tile = blockIdx.x + it * gridDim.x;
      if (u > 0) mbar_wait_sleep(smem_u32(&xc_empty[b]), (u - 1) & 1, 64);
      float *xcb = xc + (size_t)b * DP * FM;
      for (int e = lane; e < FM * DP; e += 32) {
        const int r_ = e & (FM - 1), j = e >> 7;
        const long long cg = tile * FM + r_;
        xcb[j * FM + r_] = (cg < prm.m && j < d) ? gen8_coord(ombo_pool_coord(prm.pool, cg, j), prm.gp.center[j], inv_ell[j]) : 0.f;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&xc_full[b]));
    }
  } else if (warp == 3) {
    // =============================== train slices + K* cache (one thread) =================
    // (a) keeps the ring of train slices NSL - 1 fresh blocks ahead of the generators: DP + 2 bulk copies of 256 B
    //     (coordinate rows, sigma_f2 alpha, |b|^2 of K-block kb) completing on s_full;
    // (b) walks the A stages in step order: a FRESH block that a later chunk needs is copied to the per-CTA cache in
    //     L2 once every local generator warp has written it (a_written), a CACHED block is streamed back into the
    //     stage (2-SM load, bytes counted on the leader's a_full together with this CTA's share of the arrivals).
    //     Either way the thread then arrives on a_empty: a stage is free once the MMA has consumed it AND the cache
    //     copy has read it.  (Measured alternatives, all slower: reloads issued by the B producer -- blocking or
    //     polling both cursors --, or by a generator thread when it passes the step.)
    if (elect_one() && !(prm.dbg & 128)) {
      long long it_s = 0; int i_s = 0;
      bool s_done = n_iter == 0;
      uint32_t sl = 0, slph = 0;
      auto slice_next = [&]() {
        while (!s_done) {
          if (i_s >= n_steps) { i_s = 0; if (++it_s == n_iter) s_done = true; continue; }
          const uint32_t w = sched[i_s++];
          if (!SW_FRESH(w)) continue;
          const int kb = SW_KB(w);
          mbar_wait_sleep(smem_u32(&s_empty[sl]), slph ^ 1, 32);
          const uint32_t full = smem_u32(&s_full[sl]);
          mbar_expect_tx(full, SLICE_BYTES);
          const uint32_t dst = smem_u32(xt + (size_t)sl * XT_STRIDE);
#pragma unroll 1
          for (int j = 0; j < DP; ++j) bulk_load(dst + j * (FK * 4), prm.gp.xs32 + (size_t)j * np + kb * FK, FK * 4, full);
          bulk_load(dst + DP * (FK * 4), prm.gp.alpha32 + kb * FK, FK * 4, full);
          bulk_load(dst + (DP + 1) * (FK * 4), prm.gp.b2_32 + kb * FK, FK * 4, full);
          if (++sl == NSL) { sl = 0; slph ^= 1; }
          return;
        }
      };
      for (int k = 0; k < NSL - 1; ++k) slice_next();
      uint32_t sa = 0, pa = 0;
      uint32_t wph = 0;                          // a_written completes a phase on FRESH uses of a stage only
      const uint32_t a_full_leader0 = mapa_rank(smem_u32(&a_full[0]), 0);
      unsigned char *kc = prm.kcache + (size_t)blockIdx.x * nkb * STAGE_BYTES;
      // bulk stores of one thread complete in order: a reload of block kb waits until at most `younger` of them
      // are pending, younger = copies issued after the one of kb (store_seq, this thread's private table)
      uint32_t n_stores = 0;
      for (long long it = 0; it < n_iter; ++it) {
        for (int si = 0; si < n_steps; ++si) {
          const uint32_t w = sched[si];
          const int kb = SW_KB(w);
          if (BOUND && SW_MEAN(w)) { slice_next(); continue; }   // the block's slice only, no stage
          const uint32_t stage = smem_u32(sA + sa * STAGE_BYTES);
          if (SW_FRESH(w)) {
            slice_next();
            mbar_wait_sleep(smem_u32(&a_written[sa]), (wph >> sa) & 1, 64);
            F8_TRACE(3, kb);
            wph ^= 1u << sa;
            if (SW_STORE(w)) {
              bulk_store(kc + (size_t)kb * STAGE_BYTES, stage, STAGE_BYTES);
              store_seq[kb] = n_stores++;
              asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
            }
          } else {
            const uint32_t younger = n_stores - 1u - store_seq[kb];
            if (younger == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");
            else if (younger == 1) asm volatile("cp.async.bulk.wait_group 1;\n" ::: "memory");
            else if (younger == 2) asm volatile("cp.async.bulk.wait_group 2;\n" ::: "memory");
            else if (younger == 3) asm volatile("cp.async.bulk.wait_group 3;\n" ::: "memory");
            const uint32_t full_leader = a_full_leader0 + (uint32_t)(sa * 8);
            mbar_wait_sleep(smem_u32(&a_empty[sa]), pa ^ 1, 32);
            F8_TRACE(3, 0x40 | kb);
            mbar_expect_tx_remote(full_leader, STAGE_BYTES);
            mbar_arrive_n_remote(full_leader, GEN_WARPS - 1);
            tma_load_2d_2sm(stage, &maps.kc, full_leader, 0, (int)((blockIdx.x * nkb + kb) * 256));
          }
          mbar_arrive(smem_u32(&a_empty[sa]));
          F8_TRACE(3, 0x80 | kb);
          if (++sa == NSTA) { sa = 0; pa ^= 1; }
        }
      }
      asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");
    }
  }
  } else if (warp < 8) {
    if (GW == 16) asm volatile("setmaxnreg.dec.sync.aligned.u32 72;\n");
    // =============================== epilogue (both CTAs: own 128 candidates) =============
    const int quad = warp - 4;
    const int row = quad * 32 + lane;
    uint32_t fph = 0;
    const uint32_t t_empty_leader = mapa_rank(smem_u32(&t_empty[0]), 0);
    BestPair best;                               // fused acquisition: this thread's running arg-max
    best.v = -INFINITY; best.i = 0x7fffffffffffffffLL;
    for (long long it = 0; it < ((prm.dbg & 128) ? 0 : n_iter); ++it) {
      const long long tile = blockIdx.x + it * gridDim.x;
      const long long cg = tile * FM + row;
      // the other model's posterior of this candidate: requested now, needed after the tile's last chunk
      double mo = 0.0, vo = 1.0;
      if (fuse && cg < prm.m) {
        mo = __ldg(prm.fuse.mu_other + cg);
        if (prm.fuse.var_other) vo = __ldg(prm.fuse.var_other + cg);
      }
      double ss = 0.0;
      for (int si = 0; si < n_steps; ++si) {
        const uint32_t w = sched[si];
        for (int slot = 0; slot < 2; ++slot) {
          if (!SW_DONE(w, slot)) continue;
          const int c = SW_CHUNK(w, slot);
          mbar_wait_sleep(smem_u32(&t_full[slot]), (fph >> slot) & 1, 200);
          F8_TRACE_E(c);
          fph ^= (1u << slot);
          tc_fence_after();
          float part[4] = {0.f, 0.f, 0.f, 0.f};
          const int ncw = min(CW, np - c * CW);
#pragma unroll 1
          for (int q = 0; q < ncw / 32; ++q) {
            uint32_t v[32];
            tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(slot * CW + q * 32), v);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 32; ++e) { float f = __uint_as_float(v[e]); part[e & 3] = fmaf(f, f, part[e & 3]); }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(t_empty_leader + (uint32_t)(slot * 8));
          F8_TRACE_E(0x40 | c);
          ss += (double)((part[0] + part[1]) + (part[2] + part[3]));
        }
      }
      const double var = fmax(prm.gp.sigma_f2 - ss * prm.gp.bscale[2], prm.gp.var_floor) + prm.gp.sigma_n2;
      if (!fuse) {
        if (cg < prm.m) prm.var_out[cg] = var;
      } else {
        // K4 + K5 on the epilogue warps: the generators publish the tile's mean partials (same summation order
        // as their own mu_out store, so the fused and the unfused launch see the same FP32 mean)
        const int b = (int)(it & 1);
        mbar_wait_sleep(smem_u32(&mu_full[b]), (uint32_t)(it >> 1) & 1, 64);
        const float *mub = mu_sm + (size_t)b * 4 * FM;
        const float mu_s = gen8_mean_sum(mub[row], mub[FM + row], mub[2 * FM + row], mub[3 * FM + row]);
        if (cg < prm.m) {
          const int P = prm.fuse.n_pf;
          const bool s0 = prm.fuse.self_model == 0;
          const float r = ehvi2d_value<float>(s0 ? mu_s : (float)mo, s0 ? (float)mo : mu_s, s0 ? (float)var : (float)vo,
                                              s0 ? (float)vo : (float)var, ystr, ystr + (P + 2), P,
                                              prm.fuse.exact != 0, prm.fuse.c00, prm.fuse.c01);
          if (prm.fuse.out_acq) prm.fuse.out_acq[cg] = (double)r;
          const double val = isnan(r) ? -INFINITY : (double)r;
          const long long gi = prm.fuse.index_base + cg;
          if (better(val, gi, best.v, best.i)) { best.v = val; best.i = gi; }
        }
      }
    }
    if (fuse) {
      best = warp_best(best);
      if (lane == 0) { red_v[quad] = best.v; red_i[quad] = best.i; }
      named_bar_sync(8, 128);
      if (quad == 0 && lane == 0) {
        for (int q = 1; q < 4; ++q)
          if (better(red_v[q], red_i[q], best.v, best.i)) { best.v = red_v[q]; best.i = red_i[q]; }
        prm.fuse.partials[blockIdx.x].value = best.v;
        prm.fuse.partials[blockIdx.x].index = best.i;
      }
    }
  } else {
    if (GW == 16) asm volatile("setmaxnreg.inc.sync.aligned.u32 88;\n");
    // =============================== K1 generators ========================================
    // Warp (qq, rg): K columns 16 qq .. 16 qq + 15 of the block, candidate rows 16 R rg .. 16 R (rg + 1) - 1.
    // Even lanes own the first 8 of those columns, odd lanes the other 8; a lane pair owns rows r16 + 16 rr
    // (r16 in 0..15 from the lane bits, see below) whose coordinates stay in registers for the whole tile.  The
    // lane -> (row, column group) map makes every operand store conflict-free: an STS.128 quarter-warp covers the
    // eight 16-byte chunks of the SWIZZLE_128B atom, an STS.64 half-warp the sixteen 8-byte slots of two
    // SWIZZLE_64B rows (an 8-column group alone can only ever reach half of the banks).
    // Nothing here synchronises the generator warps with each other: slices arrive through a TMA ring, the cache
    // copy waits on a_written in another warp, the mean is reduced per row group.  Warps that share a scheduler
    // (same qq) therefore drift apart and overlap their FFMA2, MUFU and conversion phases instead of queueing for
    // the same pipe in lock-step.
    const int gt = tid - 8 * 32;
    const int gw = gt >> 5;
    const int qq = gw & 3, rg = gw >> 2;
    const int gbit = lane & 1;
    const int g = 2 * qq + gbit;                   // 8-column group of the K-block
    const int r16 = ((lane >> 1) & 3) * 2 + ((lane >> 3) & 1) + 8 * (lane >> 4);
    const int row0 = 16 * R * rg + r16;
    static_assert(GW * R == 32, "generator rows must cover the tile");
    // (the kernel function is a template parameter: a run-time branch per row splits the block body into basic
    // blocks and the scheduler cannot interleave one row's MUFU chain with the next row's FFMA2s / conversions)
    constexpr int ROWS = R;
    // swizzled store offsets of this lane's first row; its other rows are 16 apart, which leaves (row & 7) and
    // (row >> 1) & 3 -- the swizzle terms -- unchanged: row r0 + 16 rr sits exactly 2048 rr (fp16 plane) / 1024 rr (e4m3
    // planes) bytes further.  Written out as immediates of the stores: with an offset array the compiler re-derived
    // all eight offsets from the lane bits in every K-block (~85 integer instructions of 690, none in the
    // stand-alone loop of scripts/k1_loop_bench.cu).
    const uint32_t off_hi0 = (uint32_t)((row0 >> 3) * 1024 + (row0 & 7) * 128 + (((g ^ (row0 & 7)) & 7) << 4));
    const uint32_t off_c80 = (uint32_t)((row0 >> 3) * 512 + (row0 & 7) * 64 + ((((g >> 1) ^ (row0 >> 1)) & 3) << 4) + (g & 1) * 8);
    const uint32_t sA_u = smem_u32(sA);
    const uint32_t a_empty_u = smem_u32(a_empty), a_written_u = smem_u32(a_written);
    const uint32_t s_full_u = smem_u32(s_full), s_empty_u = smem_u32(s_empty);
    const uint32_t a_full_leader0 = mapa_rank(smem_u32(&a_full[0]), 0);
    uint32_t sa = 0, pa = 0, sl = 0, slph = 0;
#if F8_TRACING
    const int trole = (lane == 0) ? (gw == 0 ? 5 : (gw == 5 ? 6 : (gw == GW - 1 ? 7 : -1))) : -1;
#endif
    if (prm.dbg & 8) __nanosleep(400u * (unsigned)rg);       // experiment: start the row groups out of phase
    // timing experiment (results are garbage): bit 7 = the generator loop alone, every other role idle and no barrier
    // traffic except the candidate coordinates; bit 8 = without the proxy fence as well
    const bool solo = (prm.dbg & 128) != 0;
    for (long long it = 0; it < n_iter; ++it) {
      const long long tile = blockIdx.x + it * gridDim.x;
      const int b = (int)(it & 1);
      mbar_wait_sleep(smem_u32(&xc_full[b]), (uint32_t)(it >> 1) & 1, 64);     // xc[b] holds this tile
      const float *xcb = xc + (size_t)b * DP * FM;
      float mu_acc[ROWS];
      float x[ROWS][DP], a2[ROWS];
#pragma unroll
      for (int rr = 0; rr < ROWS; ++rr) {
        mu_acc[rr] = 0.f;
        a2[rr] = gen8_load_row<DP>(xcb + row0 + 16 * rr, FM, x[rr]);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&xc_empty[b]));                   // xc[b] may be refilled
      // the K1 math of one K-block (gen8.cuh) is shared by the full and the mean-only steps -- the same operations in
      // the same order, so both see the same k' and accumulate the same mean
      {
        for (int si = 0; si < n_steps; ++si) {
          const uint32_t w = sched[si];
          const int kb = SW_KB(w);
          if (!SW_FRESH(w)) {
            // a K* block streamed back from the cache (by warp 3).  Every generator warp still waits for the stage's
            // release: a warp that skipped ahead through a run of reloads would get more than one barrier
            // phase ahead of the MMA, and a parity wait cannot tell phases two apart.
            if (!solo) mbar_wait_sleep(a_empty_u + sa * 8, pa ^ 1, 128);
            if (++sa == NSTA) { sa = 0; pa ^= 1; }
            continue;
          }
          if (BOUND && SW_MEAN(w)) {
            // a block beyond the bound: k' and the mean only -- no operands, no stage, only the slice to release
            if (!solo) mbar_wait_sleep(s_full_u + sl * 8, slph, 20);
            const float *xs = xt + sl * XT_STRIDE + 8 * g;
            float2 r2[ROWS][4];
            gen8_dist2<DP, ROWS>(xs, x, a2, r2);
            const float4 al0 = *(const float4 *)(xs + DP * FK);
            const float4 al1 = *(const float4 *)(xs + DP * FK + 4);
#pragma unroll
            for (int rr = 0; rr < ROWS; ++rr) {
              float2 kv[4];
              gen8_kval<MATERN>(r2[rr], kv);
              gen8_mean_add(kv, al0, al1, mu_acc[rr]);
            }
            __syncwarp();
            if (lane == 0 && !solo) mbar_arrive(s_empty_u + sl * 8);
            if (++sl == NSL) { sl = 0; slph ^= 1; }
            continue;
          }
          F8_TRACE_G(kb);
          if (!solo) mbar_wait_sleep(s_full_u + sl * 8, slph, 20);            // this block's train slice has landed
          F8_TRACE_G(0x40 | kb);
          const float *xs = xt + sl * XT_STRIDE + 8 * g;
          const uint32_t st_u = sA_u + sa * STAGE_BYTES;
          const uint32_t st_hi = st_u + off_hi0, st_c8 = st_u + off_c80;
          if (!(prm.dbg & 2)) {
            float2 r2[ROWS][4];
            gen8_dist2<DP, ROWS>(xs, x, a2, r2);
            const float4 al0 = *(const float4 *)(xs + DP * FK);
            const float4 al1 = *(const float4 *)(xs + DP * FK + 4);
            F8_TRACE_G(0x80 | kb);
            if (!solo) mbar_wait_sleep(a_empty_u + sa * 8, pa ^ 1, 32);        // stage released (MMA + cache copy)
            F8_TRACE_G(0xC0 | kb);
#pragma unroll
            for (int rr = 0; rr < ROWS; ++rr) {
              float2 kv[4];
              gen8_kval<MATERN>(r2[rr], kv);
              gen8_mean_add(kv, al0, al1, mu_acc[rr]);
              uint32_t hi[4];
              uint32_t c1[2], c2[2];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const __half2 h = __float22half2_rn(kv[e]);
                const float2 hf = __half22float2(h);
                // 2^12 (k' - hi): the residual is exact in FP32, the scaling too
                const float2 res = __ffma2_rn(hf, make_float2(-4096.0f, -4096.0f), __fmul2_rn(kv[e], make_float2(4096.0f, 4096.0f)));
                hi[e] = *reinterpret_cast<const uint32_t *>(&h);
                const uint32_t l8 = (uint32_t)__nv_cvt_float2_to_fp8x2(res, __NV_SATFINITE, __NV_E4M3);
                const uint32_t a8 = (uint32_t)__nv_cvt_float2_to_fp8x2(hf, __NV_SATFINITE, __NV_E4M3);
                if (e & 1) { c1[e >> 1] |= l8 << 16; c2[e >> 1] |= a8 << 16; }
                else { c1[e >> 1] = l8; c2[e >> 1] = a8; }
              }
              // (rr is a compile-time index of the unrolled row loop)
              if (rr == 0) { sts128_at<0>(st_hi, hi[0], hi[1], hi[2], hi[3]); sts64_at<F8_OFF_C1>(st_c8, c1[0], c1[1]); sts64_at<F8_OFF_C2>(st_c8, c2[0], c2[1]); }
              else if (rr == 1) { sts128_at<2048>(st_hi, hi[0], hi[1], hi[2], hi[3]); sts64_at<F8_OFF_C1 + 1024>(st_c8, c1[0], c1[1]); sts64_at<F8_OFF_C2 + 1024>(st_c8, c2[0], c2[1]); }
              else if (rr == 2) { sts128_at<4096>(st_hi, hi[0], hi[1], hi[2], hi[3]); sts64_at<F8_OFF_C1 + 2048>(st_c8, c1[0], c1[1]); sts64_at<F8_OFF_C2 + 2048>(st_c8, c2[0], c2[1]); }
              else { sts128_at<6144>(st_hi, hi[0], hi[1], hi[2], hi[3]); sts64_at<F8_OFF_C1 + 3072>(st_c8, c1[0], c1[1]); sts64_at<F8_OFF_C2 + 3072>(st_c8, c2[0], c2[1]); }
            }
          } else {
            mbar_wait_sleep(a_empty_u + sa * 8, pa ^ 1, 32);
          }
          if (!(prm.dbg & 256)) fence_proxy_async_smem();
          __syncwarp();
          F8_TRACE_G(0x20 | kb);
          if (lane == 0 && !solo) {
            mbar_arrive(s_empty_u + sl * 8);                                   // slice free
            mbar_arrive_remote(a_full_leader0 + sa * 8);                       // the leader's MMA consumes both halves
            mbar_arrive(a_written_u + sa * 8);                                 // this CTA's cache copy may start
          }
          if (++sa == NSTA) { sa = 0; pa ^= 1; }
          if (++sl == NSL) { sl = 0; slph ^= 1; }
        }
      }
      // mean: lane pairs hold the two column groups of a row, the four warps of a row group the four column pairs
      float *mub = mu_sm + (size_t)b * 4 * FM;
#pragma unroll
      for (int rr = 0; rr < ROWS; ++rr) {
        const float m = mu_acc[rr] + __shfl_xor_sync(0xffffffffu, mu_acc[rr], 1);
        if (!gbit) mub[qq * FM + row0 + 16 * rr] = m;
      }
      if (fuse) {                                  // the epilogue warps finish the mean themselves; no mu_out store
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&mu_full[b]));
        continue;
      }
      named_bar_sync(1 + rg, 128);
      const int tg = qq * 32 + lane;
      if (tg < 16 * R) {
        const int row = 16 * R * rg + tg;
        const long long cg = tile * FM + row;
        if (cg < prm.m) prm.mu_out[cg] = (double)gen8_mean_sum(mub[row], mub[FM + row], mub[2 * FM + row], mub[3 * FM + row]);
      }
      // mu_sm is double buffered by tile: the rows of buffer b are rewritten two tiles later, after the next
      // tile's barrier of the same row group
    }
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();          // nobody exits while the peer may still signal it
  if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512u));
}

// ---- host side ------------------------------------------------------------------------------
// Step schedule of one tile (see the header).  max_run <= 0: the PASS schedule (default, below).  max_run >= 1: the
// ROLLING schedule (OMBO_F8_MAXRUN, experimental).  bound_chunks >= 1: the BOUND schedule of the pass schedule (below).  The generators deliver block f = 0 .. nkb-1 in order, one per `tg`
// units of MMA time (unit = one 256-column chunk x one 64-deep K-block x the three products).  Two TMEM slots; a
// chunk opens in the slot that frees, with the already generated blocks it needs queued as reloads.  Reloads are
// issued (a) when a chunk needs no further fresh block and only its queue keeps its slot busy, (b) in the MMA time
// a fresh step leaves over (tg - its units, at most one unit banked; never more than max_run in a row), (c) at the end.  A reload that both open
// chunks still need serves both (one stage fill, two units).
void f8_build_schedule(int np, double tg, int max_run, std::vector<unsigned int> &steps, int bound_chunks) {
  const int nkb = np / FK, n_chunks = (np + 255) / 256;
  auto last_kb = [&](int c) { return std::min(4 * c + 3, nkb - 1); };
  if (bound_chunks > 0) {
    // BOUND schedule: chunks 0 .. bound_chunks - 1 (1 = chunk 0, 2 = both chunks of pass 0) take exactly the steps,
    // N-shrink and order of the pass schedule, so their accumulators -- and the epilogue's partial sums of V^2 --
    // are bit-identical to a full launch's.  The K-blocks beyond them are generated for the mean only (MEAN steps:
    // fresh, no chunk).  Nothing is reloaded, so nothing is stored.
    std::vector<unsigned int> full;
    f8_build_schedule(np, tg, 0, full, 0);
    const int nb = std::min(nkb, 4 * bound_chunks);
    steps.clear();
    for (unsigned int w : full) {
      if (!((w >> 8) & 1u) || (int)(w & 0xFFu) >= nb) continue;      // pass 0 generates blocks 0 .. 7 in order
      w &= ~(1u << 9);
      for (int sl = 0; sl < 2; ++sl)
        if ((int)((w >> (10 + 6 * sl)) & 63u) - 1 >= bound_chunks)
          w &= ~((63u << (10 + 6 * sl)) | (1u << (22 + sl)) | (1u << (24 + sl)));
      steps.push_back(w);
    }
    for (int kb = nb; kb < nkb; ++kb) steps.push_back((unsigned int)kb | (1u << 8) | (1u << 26));
    return;
  }
  if (max_run <= 0) {
    // PASS schedule (the default, measured faster on the three-stage A ring -- DESIGN.md section 4): chunks 2p and
    // 2p+1 share pass p; the blocks earlier passes generated come back as reloads that serve BOTH chunks (two units
    // per stage fill) and alternate with the pass's fresh blocks (F C F C ...), so that the generators work on the
    // next fresh block while the tensor core multiplies a reloaded one.
    steps.clear();
    for (int c0 = 0, cached = 0; c0 < n_chunks; c0 += 2) {
      const int c1 = c0 + 1 < n_chunks ? c0 + 1 : -1;
      const int end = last_kb(c1 >= 0 ? c1 : c0) + 1, nf = end - cached, nc = cached, nmin = std::min(nf, nc);
      const size_t first = steps.size();
      for (int i = 0; i < end; ++i) {
        int kb;
        if (i < 2 * nmin) kb = (i & 1) ? (i >> 1) : cached + (i >> 1);
        else kb = nf > nc ? cached + (i - nc) : (i - nf);
        unsigned int w = (unsigned int)kb | (kb >= cached ? 1u << 8 : 0u);
        if (kb <= last_kb(c0)) w |= (unsigned int)(c0 + 1) << 10;
        if (c1 >= 0) w |= (unsigned int)(c1 + 1) << 16;
        steps.push_back(w);
      }
      // FIRST on each chunk's first step of the pass, DONE on its last
      for (int s = 0; s < 2; ++s) {
        long fi = -1, la = -1;
        for (size_t i = first; i < steps.size(); ++i)
          if ((steps[i] >> (10 + 6 * s)) & 63u) { if (fi < 0) fi = (long)i; la = (long)i; }
        if (fi >= 0) { steps[fi] |= 1u << (22 + s); steps[la] |= 1u << (24 + s); }
      }
      cached = end;
    }
    std::vector<char> reloaded(nkb, 0);
    for (unsigned int w : steps) if (!((w >> 8) & 1u)) reloaded[w & 0xFFu] = 1;
    for (unsigned int &w : steps) if (((w >> 8) & 1u) && reloaded[w & 0xFFu]) w |= 1u << 9;
    return;
  }
  auto units = [&](int c, int kb) {
    const int r0 = std::max(0, kb - 4 * c) * 64;
    return (std::min(256, np - c * 256) - r0) / 256.0;
  };
  int slot_c[2] = {-1, -1};
  bool started[2] = {false, false};
  std::deque<int> pend[2];
  int next_c = 0, gen = -1;
  steps.clear();
  auto open_slot = [&](int s) {
    pend[s].clear();
    started[s] = false;
    if (next_c >= n_chunks) { slot_c[s] = -1; return; }
    const int c = next_c++;
    slot_c[s] = c;
    for (int k = 0; k <= std::min(gen, last_kb(c)); ++k) pend[s].push_back(k);
  };
  auto done = [&](int s) { return slot_c[s] >= 0 && pend[s].empty() && gen >= last_kb(slot_c[s]); };
  auto any_pend = [&]() { return (slot_c[0] >= 0 && !pend[0].empty()) || (slot_c[1] >= 0 && !pend[1].empty()); };
  auto add_chunk = [&](unsigned int &w, int s, int kb, double &u, bool (&fin)[2]) {
    w |= (unsigned int)(slot_c[s] + 1) << (10 + 6 * s);
    if (!started[s]) { w |= 1u << (22 + s); started[s] = true; }
    u += units(slot_c[s], kb);
    if (done(s)) { w |= 1u << (24 + s); fin[s] = true; }
  };
  auto emit_cached = [&]() {
    int sp = -1;
    for (int s = 0; s < 2; ++s)
      if (slot_c[s] >= 0 && !pend[s].empty() && (sp < 0 || slot_c[s] < slot_c[sp])) sp = s;
    const int kb = pend[sp].front();
    unsigned int w = (unsigned int)kb;
    double u = 0.0;
    bool fin[2] = {false, false};
    for (int s = 0; s < 2; ++s)
      if (slot_c[s] >= 0 && !pend[s].empty() && pend[s].front() == kb) {
        pend[s].pop_front();
        add_chunk(w, s, kb, u, fin);
      }
    steps.push_back(w);
    for (int s = 0; s < 2; ++s) if (fin[s]) open_slot(s);
    return u;
  };
  open_slot(0);
  open_slot(1);
  double carry = 0.0;
  for (int f = 0; f < nkb; ++f) {
    // a chunk that needs no further fresh block holds its slot only for its reloads: finish them first
    for (;;) {
      bool stuck = false;
      for (int s = 0; s < 2; ++s) stuck |= slot_c[s] >= 0 && last_kb(slot_c[s]) < f && !pend[s].empty();
      if (!stuck) break;
      carry -= emit_cached();
    }
    gen = f;
    unsigned int w = (unsigned int)f | (1u << 8);
    double u = 0.0;
    bool fin[2] = {false, false};
    for (int s = 0; s < 2; ++s)
      if (slot_c[s] >= 0 && f <= last_kb(slot_c[s])) add_chunk(w, s, f, u, fin);
    steps.push_back(w);
    for (int s = 0; s < 2; ++s) if (fin[s]) open_slot(s);
    // at most max_run reloads in a row: the A ring is three stages deep, and a longer run of reloads would hold
    // the stage the generators need for the second half of their next block
    double budget = carry + tg - u;
    for (int run = 0; run < max_run && budget > 0.0 && any_pend(); ++run) budget -= emit_cached();
    carry = std::min(budget, 1.0);
  }
  while (any_pend()) emit_cached();
  // fresh blocks that some later step reloads have to be copied to the cache
  std::vector<char> reloaded(nkb, 0);
  for (unsigned int w : steps) if (!((w >> 8) & 1u)) reloaded[w & 0xFFu] = 1;
  for (unsigned int &w : steps) if (((w >> 8) & 1u) && reloaded[w & 0xFFu]) w |= 1u << 9;
}

// debug / test hook (not part of the public header): the schedule for n_pad as the kernel will walk it
extern "C" int ombo_debug_f8_schedule(int n_pad, double tg, int max_run, unsigned int *out, int cap) {
  std::vector<unsigned int> steps;
  f8_build_schedule(n_pad, tg, max_run, steps, 0);
  for (int i = 0; i < (int)steps.size() && i < cap; ++i) out[i] = steps[i];
  return (int)steps.size();
}
extern "C" int ombo_debug_f8_bound_schedule(int n_pad, int bound_chunks, unsigned int *out, int cap) {
  std::vector<unsigned int> steps;
  f8_build_schedule(n_pad, 3.0, 0, steps, bound_chunks < 1 ? 1 : bound_chunks);
  for (int i = 0; i < (int)steps.size() && i < cap; ++i) out[i] = steps[i];
  return (int)steps.size();
}

static int make_plane_map(CUtensorMap *map, const void *base, int n_pad, int esz, int box_rows) {
  PFN_encodeTiled_t enc = ombo_get_encode_tiled();
  if (!enc) { ombo_set_error("cuTensorMapEncodeTiled is not available from the driver"); return OMBO_ERR_CUDA; }
  cuuint64_t dims[2] = {(cuuint64_t)n_pad, (cuuint64_t)n_pad};
  cuuint64_t strides[1] = {(cuuint64_t)n_pad * esz};
  cuuint32_t box[2] = {FK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, esz == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(base),
                   dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   esz == 2 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { ombo_set_error("cuTensorMapEncodeTiled (f8c plane) failed (%d)", (int)r); return OMBO_ERR_CUDA; }
  return OMBO_OK;
}

// dynamic shared memory without the step schedule and the fused stripes: operand rings, candidate coordinates,
// train slices, mean partials, barriers + tables (see the carve-up at the top of the kernel), alignment slack
static size_t f8_smem_base(int DP) {
  return (size_t)6 * STAGE_BYTES + 2 * (size_t)DP * FM * 4 + (size_t)F8_NSL * (DP + 2) * FK * 4 + 8 * FM * 4 + 16 +
         34 * 8 + 16 * 8 + 128 * 4 + 16 + 2 * 8 + 8 * 8 + 1024;
}

template <int DP, int R, int GW, bool MATERN, bool BOUND>
static int launch_fast8(ombo_ctx *ctx, const F8Maps &maps, FastParams prm, int grid, cudaStream_t s) {
  // the fused stripes first, then the schedule if it still fits (the same order as the can-fuse test of the caller)
  size_t smem = f8_smem_base(DP) + (prm.fuse.on ? (size_t)2 * (prm.fuse.n_pf + 2) * 4 : 0);
  prm.sched_in_smem = smem + (size_t)prm.n_steps * 4 <= 227 * 1024 ? 1 : 0;
  if (prm.sched_in_smem) smem += (size_t)prm.n_steps * 4;
  // per device, not per process: the attribute belongs to the (function, device) pair
  OMBO_CUDA(cudaFuncSetAttribute(k_posterior_fast8<DP, R, GW, MATERN, BOUND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ProfScope prof(ctx, s);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3((8 + GW) * 32);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  OMBO_CUDA(cudaLaunchKernelEx(&cfg, k_posterior_fast8<DP, R, GW, MATERN, BOUND>, maps, prm));
  return OMBO_OK;
}

// the step schedule of a tile for n_pad (full, or bound with bound_chunks chunks), built and uploaded once
static int f8_schedule(ombo_ctx *ctx, int n_pad, int bound_chunks, cudaStream_t s) {
  const int k = bound_chunks > 0 ? 1 : 0;
  if (ctx->f8_sched_np[k] == n_pad && ctx->f8_sched_depth[k] == bound_chunks) return OMBO_OK;
  std::vector<unsigned int> steps;
  f8_build_schedule(n_pad, ctx->knobs.f8_tg, ctx->knobs.f8_max_run, steps, bound_chunks);
  if ((int)steps.size() > ctx->f8_sched_cap[k]) {
    if (ctx->f8_sched[k]) OMBO_CUDA(cudaFree(ctx->f8_sched[k]));
    ctx->f8_sched[k] = nullptr;
    OMBO_CUDA(cudaMalloc(&ctx->f8_sched[k], steps.size() * sizeof(unsigned int)));
    ctx->f8_sched_cap[k] = (int)steps.size();
  }
  OMBO_CUDA(cudaStreamSynchronize(s));            // a launch in flight may still read the old table
  OMBO_CUDA(cudaMemcpy(ctx->f8_sched[k], steps.data(), steps.size() * sizeof(unsigned int), cudaMemcpyHostToDevice));
  ctx->f8_sched_np[k] = n_pad;
  ctx->f8_sched_depth[k] = bound_chunks;
  ctx->f8_sched_len[k] = (int)steps.size();
  return OMBO_OK;
}

// shared memory of a fused launch: the stripes must fit beside the operand rings (the schedule may stay in global memory)
static bool f8_fuse_fits(const GpDev &gp, int n_pf, int n_steps) {
  const int dp = gp.d <= 2 ? 2 : (gp.d + 1) / 2 * 2;
  size_t need = f8_smem_base(dp) + (size_t)2 * (n_pf + 2) * 4;
  if (need + (size_t)n_steps * 4 <= 227 * 1024) need += (size_t)n_steps * 4;
  return need <= 227 * 1024;
}

bool ombo_f8_can_fuse(ombo_ctx *ctx, const GpDev &gp, int n_pf, int bound_chunks, cudaStream_t s) {
  if (f8_schedule(ctx, gp.n_pad, bound_chunks, s)) return false;
  return f8_fuse_fits(gp, n_pf, ctx->f8_sched_len[bound_chunks > 0 ? 1 : 0]);
}

// mu / var of one GP whose planes are in the f8c format (gp.flags & OMBO_GP_F8C_PLANES), d <= 12
int ombo_posterior_fast8(ombo_ctx *ctx, const GpDev &gp, const PoolDev &pool, long long m, double *mu, double *var,
                         cudaStream_t s, const FuseAcq *fuse_req, int *fused, int bound_chunks) {
  if (fused) *fused = 0;
  const long long tiles = (m + FM - 1) / FM;
  F8Maps maps;
  const unsigned char *c1 = (const unsigned char *)gp.blo, *c2 = c1 + (size_t)gp.n_pad * gp.n_pad;
  int rc;
  if ((rc = make_plane_map(&maps.hi128, gp.bhi, gp.n_pad, 2, 128))) return rc;
  if ((rc = make_plane_map(&maps.hi32, gp.bhi, gp.n_pad, 2, 32))) return rc;
  if ((rc = make_plane_map(&maps.c1_128, c1, gp.n_pad, 1, 128))) return rc;
  if ((rc = make_plane_map(&maps.c1_32, c1, gp.n_pad, 1, 32))) return rc;
  if ((rc = make_plane_map(&maps.c2_128, c2, gp.n_pad, 1, 128))) return rc;
  if ((rc = make_plane_map(&maps.c2_32, c2, gp.n_pad, 1, 32))) return rc;
  maps.kc = maps.hi128;
  FastParams prm;
  prm.gp = gp; prm.pool = pool; prm.m = m; prm.mu_out = mu; prm.var_out = var;
  prm.dbg = ctx->knobs.fast_dbg; prm.kcache = nullptr;
  const bool want_prof = ctx->knobs.fast_profile != 0;
  if (want_prof && !ctx->prof_dev) OMBO_CUDA(cudaMalloc(&ctx->prof_dev, 16 * 256 * sizeof(long long)));
  prm.prof = want_prof ? ctx->prof_dev : nullptr;
  prm.trace = nullptr;
  static long long *trace_dev = nullptr;
  if (ctx->knobs.fast_profile == 2) {
    if (!trace_dev) OMBO_CUDA(cudaMalloc(&trace_dev, 8 * F8_TRACE_N * sizeof(long long)));
    OMBO_CUDA(cudaMemsetAsync(trace_dev, 0, 8 * F8_TRACE_N * sizeof(long long), s));
    prm.trace = trace_dev;
  }
  if (want_prof) OMBO_CUDA(cudaMemsetAsync(ctx->prof_dev, 0, 16 * 256 * sizeof(long long), s));
  int grid = (int)(tiles < ctx->num_sms ? tiles : ctx->num_sms);
  grid = (grid + 1) / 2 * 2;                    // whole pairs; a surplus CTA runs a dummy tile
  if (grid > ctx->num_sms) grid = ctx->num_sms / 2 * 2;
  // step schedule of a tile: a function of n_pad, the bound depth (and the knobs) only
  const int sk = bound_chunks > 0 ? 1 : 0;
  if ((rc = f8_schedule(ctx, gp.n_pad, bound_chunks, s))) return rc;
  prm.sched = ctx->f8_sched[sk];
  prm.n_steps = ctx->f8_sched_len[sk];
  prm.fuse.on = 0;
  if (fuse_req) {
    // fused 2-D EHVI + arg-max: only while the stripes fit beside everything else in shared memory
    if (f8_fuse_fits(gp, fuse_req->n_pf, prm.n_steps)) {
      rc = ombo_ws_reserve(&ctx->ws_partial, &ctx->ws_partial_bytes, (size_t)grid * sizeof(ombo_best));
      if (rc) return rc;
      prm.fuse = *fuse_req;
      prm.fuse.on = 1;
      prm.fuse.partials = (ombo_best *)ctx->ws_partial;
      if (fused) *fused = grid;
    }
  }
  if (gp.n_pad > 512 && !bound_chunks) {         // more than two chunks: generated K* blocks are cached in L2 for later chunks
    rc = ombo_ws_reserve(&ctx->ws_scratch, &ctx->ws_scratch_bytes, (size_t)grid * (gp.n_pad / FK) * STAGE_BYTES);
    if (rc) return rc;
    prm.kcache = (unsigned char *)ctx->ws_scratch;
    rc = ombo_make_linear_map(&maps.kc, prm.kcache, (size_t)grid * (gp.n_pad / FK) * 256);
    if (rc) return rc;
  }
  const int d = gp.d;
  // the bound schedule leaves the generators alone on the critical path, below the power cap: 16 warps (measured,
  // DESIGN.md section 4); the full schedule keeps 8 unless OMBO_FAST_GEN_WARPS says otherwise
  const int gw_knob = ctx->knobs.fast_gen_warps;
  const bool gw16 = gw_knob ? gw_knob == 16 : bound_chunks > 0;
  const bool mat = gp.kernel == OMBO_KERNEL_MATERN52;
#define F8_LAUNCH(DPV, RV, GWV, BV)                                                                                  \
  (mat ? launch_fast8<DPV, RV, GWV, true, BV>(ctx, maps, prm, grid, s) : launch_fast8<DPV, RV, GWV, false, BV>(ctx, maps, prm, grid, s))
#define F8_DISPATCH(DPV)                                                                                             \
  rc = bound_chunks ? (gw16 ? F8_LAUNCH(DPV, 2, 16, true) : F8_LAUNCH(DPV, 4, 8, true))                               \
                    : (gw16 ? F8_LAUNCH(DPV, 2, 16, false) : F8_LAUNCH(DPV, 4, 8, false))
  if (d <= 2) { F8_DISPATCH(2); }
  else if (d <= 4) { F8_DISPATCH(4); }
  else if (d <= 6) { F8_DISPATCH(6); }
  else if (d <= 8) { F8_DISPATCH(8); }
  else if (d <= 10) { F8_DISPATCH(10); }
  else { F8_DISPATCH(12); }
#undef F8_DISPATCH
#undef F8_LAUNCH
  if (rc) return rc;
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  if (want_prof) {
    static long long h[16 * 256];
    OMBO_CUDA(cudaStreamSynchronize(s));
    OMBO_CUDA(cudaMemcpy(h, ctx->prof_dev, sizeof(h), cudaMemcpyDeviceToHost));
    double a[8] = {0};
    for (int b = 0; b < grid; ++b) for (int k = 0; k < 8; ++k) a[k] += (double)h[b * 16 + k] / grid;
    if (prm.trace) {
      static long long ht[8 * F8_TRACE_N];
      OMBO_CUDA(cudaMemcpy(ht, prm.trace, sizeof(ht), cudaMemcpyDeviceToHost));
      const char *path = getenv("OMBO_FAST_TRACE_FILE");
      FILE *f = fopen(path ? path : "gpurun_out/fast8_trace.txt", "w");
      if (f) {
        for (int r = 0; r < 8; ++r)
          for (int e = 0; e < F8_TRACE_N && ht[r * F8_TRACE_N + e]; ++e)
            fprintf(f, "%d %lld %lld\n", r, ht[r * F8_TRACE_N + e] >> 8, ht[r * F8_TRACE_N + e] & 255);
        fclose(f);
      }
    }
    fprintf(stderr, "[fast8 prof] per-CTA cycles (leader + peer averaged): tma.wait_b_empty %.0f / tma.total %.0f | mma.wait_a_full %.0f "
            "wait_b_full %.0f wait_t_empty %.0f | gen.wait_a_empty %.0f  (tiles/CTA %.1f)\n",
            a[0], a[1], 2 * a[2], 2 * a[3], 2 * a[4], a[5], (double)tiles / grid);
  }
  return OMBO_OK;
}
