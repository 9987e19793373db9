// K1 + K2, fast mode: bf16x3 split-precision on the 5th-gen tensor cores (tcgen05 + TMEM + TMA).
// Same contract as posterior_fp64.cu (mu, var per candidate for one GP), tolerance rtol 1e-3.
//
//   V = K* . (sigma_f2 L^-1)^T     K* = k'(r) in (0,1] generated ON CHIP, never touching HBM
//   A = K*  = A_hi + A_lo,  B = s sigma_f2 L^-1 = B_hi + B_lo (16-bit planes from K3: bf16, or scaled fp16 for
//   ill-conditioned GPs -- template parameter F16, selected from ombo_gp.reserved)
//   V ~= A_hi B_hi^T + A_lo B_hi^T + A_hi B_lo^T      (three kind::f16 MMAs, FP32 accumulate in TMEM)
//   var = sigma_f2 - sum_j V_j^2 (V = L^-1 k*),  mu = sum_i k'_i (sigma_f2 alpha_i) on the CUDA cores.
//
// One persistent CTA per SM owns a tile of 128 candidates (UMMA M = 128, cta_group::1), 256-column accumulator chunks:
//   warp 0      TMA producer: 256x64 16-bit planes of B (SWIZZLE_128B) into a 3-entry ring, one plane per entry
//               (hi, then lo: the lo plane of a unit can still be in flight while its hi plane is multiplied);
//               on the diagonal K-blocks only the rows of the band are fetched
//   warp 1      MMA issuer (one elected lane): 12 tcgen05.mma (4 k-steps x 3 products) per (chunk, K-block),
//               N shrinking 256/192/128/64 on the diagonal K-blocks
//   warp 2      TMEM allocator (512 columns = 2 accumulator chunks of 256 columns)
//   warps 4-7   epilogue: tcgen05.ld 32x32b (one candidate row per thread), square + row-sum
//   warps 8-15  K1 generators: r^2 = |a|^2 + |b|^2 - 2 a.b on centred scaled inputs (packed FFMA2),
//               Matern-5/2 / RBF via MUFU (sqrt, ex2), bf16 hi/lo split, written straight into the UMMA
//               K-major SWIZZLE_128B operand layout in shared memory (3-stage ring), and the mean.
// L^-1 is lower triangular: chunk c only needs K-blocks kb <= 4c+3, the rest is never loaded nor multiplied.
// TMEM holds 2 chunks, so n_pad <= 512 is one pass; larger n takes several passes and the K* blocks generated
// by a pass are copied to a per-CTA cache in L2 (bulk store of the 32 KB stage) and streamed back by a bulk
// load in the later passes: every K* block is generated exactly once per tile.
// Within a pass the loop is K-outer, so a chunk's accumulator completes as soon as the K loop crosses
// its diagonal and the epilogue drains it while the tensor core continues on the later chunks.
// The UMMA runs at its N/2-cycle floor (scripts/umma_bench.cu); what limits this kernel is shared-memory traffic
// per MAC (the A tile is re-read by every MMA: 32 B/clk at N = 256, on top of 64 B/clk of B reads and the TMA / K1
// writes) and, at the power cap, issued work -- hence 256-column chunks on one CTA, with N shrinking on the diagonal
// (a cta_group::2 pair halves the B traffic but cannot shrink N and was slower at the cap: DESIGN.md section 4).
// PTX wrappers and the parameter block: umma.cuh.
#include "umma.cuh"


// DP  = input dimension padded to the instantiated size (padding coordinates are zero on both sides)
// R   = candidate rows held in registers per generator thread (4 when DP <= 12, else 2)
// F16 = fp16 planes (ill-conditioned GP): fp16 hi/lo split of K* and direct distances
template <int DP, int R, bool F16>
__global__ void __launch_bounds__(16 * 32, 1)
k_posterior_fast(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo,
                 const __grid_constant__ CUtensorMap map_kc, const FastParams prm) {
  constexpr int NSTA = 3, NSTB = 3;               // ring depths (32 KB entries, 192 KB in all)
  constexpr int GEN_WARPS = 8, GEN_THREADS = GEN_WARPS * 32;
  constexpr int CW = 256;                        // accumulator chunk width = widest UMMA N
  constexpr int NSLOT = 512 / CW;                // TMEM accumulator slots
  constexpr int KSH = 2;                         // chunk c needs K-blocks kb < (c + 1) << KSH
  constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(CW >> 3) << 17) | ((uint32_t)(FM >> 4) << 24);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int d = prm.gp.d, np = prm.gp.n_pad;
  const int nkb = np / FK;
  const int n_chunks = (np + CW - 1) / CW;
  const int n_pass = (n_chunks + NSLOT - 1) / NSLOT;
  const long long n_tiles = (prm.m + FM - 1) / FM;
  const long long n_iter = (n_tiles + gridDim.x - 1) / gridDim.x;
  auto last_kb = [&](int c) { return min(((c + 1) << KSH) - 1, nkb - 1); };

  // ---- shared memory carve-up ----
  unsigned char *sA = fast_smem + ((1024u - (smem_u32(fast_smem) & 1023u)) & 1023u);   // SWIZZLE_128B: 1024-B aligned
  unsigned char *sB = sA + NSTA * STAGE_BYTES;                 // NSTB x one plane of a 256-row B tile (32 KB)
  float *xc = (float *)(sB + NSTB * STAGE_BYTES);              // [DP][128] scaled candidate coords
  float *xt = xc + (size_t)DP * FM;                            // [2][(DP+2)][64] train slice (+ alpha, |b|^2 rows)
  float *mu_sm = xt + 2 * (size_t)(DP + 2) * FK;               // [8][128]
  uint64_t *bars = (uint64_t *)(((uintptr_t)(mu_sm + 8 * FM) + 15) & ~(uintptr_t)15);
  uint64_t *a_full = bars, *a_empty = bars + NSTA, *b_full = bars + 2 * NSTA, *b_empty = b_full + NSTB;
  uint64_t *t_full = b_empty + NSTB, *t_empty = t_full + 4;
  uint32_t *tmem_slot = (uint32_t *)(t_empty + 4);
  double *inv_ell = (double *)(bars + 24);   // 1 / lengthscale: the per-tile coordinate prep multiplies (an FP64
                                             // division is ~14 instructions on a pipe the B200 barely has)

  if (tid == 0) {
    for (int j = 0; j < DP; ++j) inv_ell[j] = j < d ? 1.0 / prm.gp.ell[j] : 0.0;
    for (int s = 0; s < NSTA; ++s) {
      mbar_init(smem_u32(&a_full[s]), GEN_WARPS);
      mbar_init(smem_u32(&a_empty[s]), 1);
    }
    for (int s = 0; s < NSTB; ++s) {
      mbar_init(smem_u32(&b_full[s]), 1);
      mbar_init(smem_u32(&b_empty[s]), 1);
    }
    for (int s = 0; s < 4; ++s) { mbar_init(smem_u32(&t_full[s]), 1); mbar_init(smem_u32(&t_empty[s]), 4); }
    fence_mbar_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // =============================== TMA producer (B tiles) ===============================
    if (elect_one()) {
      uint32_t st = 0, ph = 0;
      long long w_bempty = 0; const bool pon = prm.prof != nullptr; const long long t_start = clock64();
      for (long long it = 0; it < n_iter; ++it) {
        for (int p = 0; p < n_pass; ++p) {
          const int c_first = NSLOT * p, c_last = min(c_first + NSLOT - 1, n_chunks - 1);
          const int kb_end = last_kb(c_last) + 1;
          for (int kb = 0; kb < kb_end; ++kb) {
            for (int c = max(c_first, kb >> KSH); c <= c_last; ++c) {
              // two ring entries per unit: the hi plane, then the lo plane.  Rows of the chunk above the diagonal
              // band are never multiplied (the UMMA's N shrinks): on the diagonal K-blocks only the 64-row boxes
              // from r0 on are fetched (a ragged last chunk keeps the per-plane maps: their out-of-bounds rows are
              // zero-filled)
              const int r0 = ((c + 1) * CW <= np) ? max(0, kb - 4 * c) * 64 : 0;
#pragma unroll
              for (int pl = 0; pl < 2; ++pl) {
                mbar_wait_prof(smem_u32(&b_empty[st]), ph ^ 1, 64, w_bempty, pon);
                const uint32_t full = smem_u32(&b_full[st]);
                const uint32_t dst = smem_u32(sB + st * STAGE_BYTES);
                if (r0 == 0) {
                  mbar_expect_tx(full, STAGE_BYTES);
                  tma_load_2d(dst, pl == 0 ? &map_hi : &map_lo, full, kb * FK, c * CW);
                } else {
                  mbar_expect_tx(full, (uint32_t)((CW - r0) * 128));
                  for (int rr = r0; rr < CW; rr += 64)       // map_kc: both planes as one (2 n_pad, n_pad) matrix, 64-row boxes
                    tma_load_2d(dst + (uint32_t)(rr * 128), &map_kc, full, kb * FK, pl * np + c * CW + rr);
                }
                if (++st == NSTB) { st = 0; ph ^= 1; }
              }
            }
          }
        }
      }
      if (pon) { prm.prof[blockIdx.x * 16 + 0] = w_bempty; prm.prof[blockIdx.x * 16 + 1] = clock64() - t_start; }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer ===========================================
    if (elect_one()) {
      uint32_t sa = 0, pa = 0, sb = 0, pb = 0, tph = 0;   // tph: per-slot phase bits of t_empty
      // operand format chosen by K3 on the device (bscale[3]): bf16 planes for well-conditioned GPs, fp16 otherwise
      constexpr uint32_t IDESC_RT = IDESC | (F16 ? 0u : ((1u << 7) | (1u << 10)));
      long long w_afull = 0, w_bfull = 0, w_tempty = 0; const bool pon = prm.prof != nullptr;
      for (long long it = 0; it < n_iter; ++it) {
        for (int p = 0; p < n_pass; ++p) {
          const int c_first = NSLOT * p, c_last = min(c_first + NSLOT - 1, n_chunks - 1);
          const int kb_end = last_kb(c_last) + 1;
          for (int kb = 0; kb < kb_end; ++kb) {
            mbar_wait_prof(smem_u32(&a_full[sa]), pa, MMA_SLEEP_NS, w_afull, pon);
            tc_fence_after();
            const uint32_t a_hi = smem_u32(sA + sa * STAGE_BYTES), a_lo = a_hi + PLANE_BYTES;
            for (int c = max(c_first, kb >> KSH); c <= c_last; ++c) {
              const int slot = c & (NSLOT - 1);
              if (kb == 0) {                                  // first touch of this accumulator slot
                mbar_wait_prof(smem_u32(&t_empty[slot]), ((tph >> slot) & 1) ^ 1, MMA_SLEEP_NS, w_tempty, pon);
                tph ^= (1u << slot);
                tc_fence_after();
              }
              // rows of the chunk above the diagonal band are zero: skip them (N = 256, 192, 128 or 64)
              const int r0 = max(0, kb - 4 * c) * 64;
              const uint32_t dcolw = tmem_base + (uint32_t)(slot * CW + r0);
              const uint32_t idw = (IDESC_RT & ~(0x3Fu << 17)) | ((uint32_t)((CW - r0) >> 3) << 17);
              // hi plane: A_hi.B_hi and A_lo.B_hi
              mbar_wait_prof(smem_u32(&b_full[sb]), pb, MMA_SLEEP_NS, w_bfull, pon);
              tc_fence_after();
              uint32_t bp = smem_u32(sB + sb * STAGE_BYTES) + (uint32_t)(r0 * 128);
#pragma unroll
              for (int ks = 0; ks < FK / 16; ++ks) {
                const uint64_t dbh = make_sdesc(bp + ks * 32);
                umma_bf16(dcolw, make_sdesc(a_hi + ks * 32), dbh, idw, (kb > 0 || ks > 0) ? 1u : 0u);
                umma_bf16(dcolw, make_sdesc(a_lo + ks * 32), dbh, idw, 1u);
              }
              umma_commit(smem_u32(&b_empty[sb]));
              if (++sb == NSTB) { sb = 0; pb ^= 1; }
              // lo plane: A_hi.B_lo
              mbar_wait_prof(smem_u32(&b_full[sb]), pb, MMA_SLEEP_NS, w_bfull, pon);
              tc_fence_after();
              bp = smem_u32(sB + sb * STAGE_BYTES) + (uint32_t)(r0 * 128);
#pragma unroll
              for (int ks = 0; ks < FK / 16; ++ks)
                umma_bf16(dcolw, make_sdesc(a_hi + ks * 32), make_sdesc(bp + ks * 32), idw, 1u);
              umma_commit(smem_u32(&b_empty[sb]));
              if (++sb == NSTB) { sb = 0; pb ^= 1; }
              if (kb == last_kb(c)) umma_commit(smem_u32(&t_full[slot]));      // chunk complete
            }
            umma_commit(smem_u32(&a_empty[sa]));
            if (++sa == NSTA) { sa = 0; pa ^= 1; }
          }
        }
      }
      if (pon) { prm.prof[blockIdx.x * 16 + 2] = w_afull; prm.prof[blockIdx.x * 16 + 3] = w_bfull; prm.prof[blockIdx.x * 16 + 4] = w_tempty; }
    }
  } else if (warp >= 4 && warp < 8) {
    // =============================== epilogue =============================================
    const int quad = warp - 4;
    const int row = quad * 32 + lane;
    uint32_t fph = 0;                                        // per-slot phase bits of t_full
    for (long long it = 0; it < n_iter; ++it) {
      const long long tile = blockIdx.x + it * gridDim.x;
      double ss = 0.0;
      for (int c = 0; c < n_chunks; ++c) {
        const int slot = c & (NSLOT - 1);
        mbar_wait_sleep(smem_u32(&t_full[slot]), (fph >> slot) & 1, 200);
        fph ^= (1u << slot);
        tc_fence_after();
        float part[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int q = 0; q < CW / 32; ++q) {
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(slot * CW + q * 32), v);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 32; ++e) { float f = __uint_as_float(v[e]); part[e & 3] = fmaf(f, f, part[e & 3]); }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&t_empty[slot]));
        ss += (double)((part[0] + part[1]) + (part[2] + part[3]));
      }
      const long long cg = tile * FM + row;
      if (cg < prm.m) {
        // V = k' (s sigma_f2 L^-1)^T = s L^-1 k*, so ss = s^2 ||L^-1 k*||^2 (s: power-of-two scale of the fp16 planes)
        double v = prm.gp.sigma_f2 - ss * prm.gp.bscale[2];
        prm.var_out[cg] = fmax(v, prm.gp.var_floor) + prm.gp.sigma_n2;
      }
    }
  } else if (warp >= 8) {
    // =============================== K1 generators ========================================
    // Warp q owns operand chunk q (K columns 8q..8q+7 of the block); lane l owns candidate rows
    // l + 32 rr.  The candidate coordinates live in registers for the whole tile, so the only
    // shared-memory reads in the inner loop are two broadcast LDS.128 of (negated) training
    // coordinates per dimension: the LSU traffic that competes with the UMMA operand fetch is
    // 1/R of a row-per-thread mapping.
    const int gt = tid - 8 * 32;                 // 0 .. 255
    const int q = gt >> 5;                       // operand chunk 0..7 of this warp
    const bool matern = (prm.gp.kernel == OMBO_KERNEL_MATERN52);
    constexpr bool f16 = F16, direct = F16;         // fp16 planes (ill-conditioned GP): fp16 split + direct distances
    constexpr int RB = 128 / (32 * R);              // row batches per K-block
    constexpr int XT_STRIDE = (DP + 2) * FK;
    uint32_t sa = 0, pa = 0;
    int xbuf = 0;
    long long w_aempty = 0, w_bar = 0; const bool pon = prm.prof != nullptr;
    // train-slice loader: 16 x 16-byte segments per row, 16 rows per sweep; rows < DP are the centred scaled
    // coordinates, row DP is sigma_f2 * alpha, row DP + 1 the squared norms |b_i|^2.  cp.async: global -> smem with no register staging, so
    // the copy of the NEXT slice really is in flight while this K-block is computed.
    constexpr int LD_ROWS = GEN_THREADS / 16;
    const int ld_j = gt >> 4, ld_o = (gt & 15) * 4;
    constexpr int LD_SWEEPS = (DP + 2 + LD_ROWS - 1) / LD_ROWS;
    auto prefetch_slice = [&](float *dst, int kb) {
#pragma unroll
      for (int sw = 0; sw < LD_SWEEPS; ++sw) {
        const int jj = ld_j + LD_ROWS * sw;
        if (jj <= DP + 1) {
          const float *src = (jj < DP) ? prm.gp.xs32 + (size_t)jj * np + kb * FK + ld_o
                                       : (jj == DP ? prm.gp.alpha32 : prm.gp.b2_32) + kb * FK + ld_o;
          const uint32_t sd = smem_u32(dst + jj * FK + ld_o);
          asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" ::"r"(sd), "l"(src) : "memory");
        }
      }
      asm volatile("cp.async.commit_group;\n" ::: "memory");
    };
    prefetch_slice(xt, 0);
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    for (long long it = 0; it < n_iter; ++it) {
      const long long tile = blockIdx.x + it * gridDim.x;
      asm volatile("bar.sync 1, %0;\n" ::"n"(GEN_THREADS));
      for (int e = gt; e < FM * DP; e += GEN_THREADS) {
        const int r_ = e & (FM - 1), j = e >> 7;
        const long long cg = tile * FM + r_;
        // -2 * centred scaled coordinate: r^2 = |a|^2 + |b|^2 + sum_j (-2 a_j) b_j
        xc[j * FM + r_] = (cg < prm.m && j < d)
                              ? -2.0f * (float)((ombo_pool_coord(prm.pool, cg, j) - prm.gp.center[j]) * inv_ell[j])
                              : 0.f;
      }
      asm volatile("bar.sync 1, %0;\n" ::"n"(GEN_THREADS));
      float mu_acc[4] = {0.f, 0.f, 0.f, 0.f};
      float x[R][DP], a2[R];                       // (-2 x) coordinates and |a|^2 of this lane's rows
      if (RB == 1) {
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
          float acc = 0.f;
#pragma unroll
          for (int j = 0; j < DP; ++j) { x[rr][j] = xc[j * FM + lane + 32 * rr]; acc = fmaf(x[rr][j], x[rr][j], acc); }
          a2[rr] = 0.25f * acc;
        }
      }
      for (int p = 0; p < n_pass; ++p) {
        const int c_last = min(NSLOT * p + NSLOT - 1, n_chunks - 1);
        const int kb_end = last_kb(c_last) + 1;
        // K* blocks generated by an earlier pass of this tile are not recomputed: they were copied to a
        // per-CTA cache in L2 (bulk store of the 32 KB operand stage) and are streamed back by a bulk load
        // that completes the stage's full barrier.  Every K* block is generated exactly once per tile.
        const bool use_cache = prm.kcache != nullptr;
        const int kb_cached = (use_cache && p > 0) ? last_kb(min(NSLOT * (p - 1) + NSLOT - 1, n_chunks - 1)) + 1 : 0;
        const bool store_cache = use_cache && (p + 1 < n_pass);
        unsigned char *kc = prm.kcache + (size_t)blockIdx.x * nkb * STAGE_BYTES;
        if (kb_cached > 0 && gt == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");   // stores landed
        for (int kb = 0; kb < kb_end; ++kb) {
          const bool do_mu = use_cache || p == n_pass - 1;     // without the cache every pass regenerates K*
          const int kb_next = (kb + 1 < kb_end) ? kb + 1 : 0;
          prefetch_slice(xt + (xbuf ^ 1) * XT_STRIDE, kb_next);          // lands while this K-block is computed
          if (kb < kb_cached) {
            if (gt == 0) {
              // ONE thread performs all GEN_WARPS arrivals of this phase, and only after the stage has been
              // released: the other warps do not wait on a_empty here, so an arrival of their own could land
              // in the still-open phase of two K-blocks ago (its bulk load may not have completed yet)
              mbar_wait_prof(smem_u32(&a_empty[sa]), pa ^ 1, 32, w_aempty, pon);
              mbar_expect_tx(smem_u32(&a_full[sa]), STAGE_BYTES);
              mbar_arrive_n(smem_u32(&a_full[sa]), GEN_WARPS - 1);
              bulk_load(smem_u32(sA + sa * STAGE_BYTES), kc + (size_t)kb * STAGE_BYTES, STAGE_BYTES, smem_u32(&a_full[sa]));
            }
            if (++sa == NSTA) { sa = 0; pa ^= 1; }
            asm volatile("cp.async.wait_group 0;\n" ::: "memory");
            asm volatile("bar.sync 1, %0;\n" ::"n"(GEN_THREADS));
            xbuf ^= 1;
            continue;
          }
          const float *xs = xt + xbuf * XT_STRIDE + 8 * q;
          unsigned char *st_hi = sA + sa * STAGE_BYTES, *st_lo = st_hi + PLANE_BYTES;
#pragma unroll 1
          for (int rb = 0; rb < RB; ++rb) {
            if (RB > 1) {
#pragma unroll
              for (int rr = 0; rr < R; ++rr) {
                float acc = 0.f;
#pragma unroll
                for (int j = 0; j < DP; ++j) {
                  x[rr][j] = xc[j * FM + lane + 32 * (R * rb + rr)];
                  acc = fmaf(x[rr][j], x[rr][j], acc);
                }
                a2[rr] = 0.25f * acc;
              }
            }
            float2 r2[R][4];
            if (direct) {
              // direct differences: (b_j - a_j)^2 summed, no |a|^2 + |b|^2 - 2 a.b cancellation (ill-conditioned GPs)
#pragma unroll
              for (int rr = 0; rr < R; ++rr)
#pragma unroll
                for (int e = 0; e < 4; ++e) r2[rr][e] = make_float2(0.f, 0.f);
#pragma unroll
              for (int j = 0; j < DP; ++j) {
                const float4 t0 = *(const float4 *)(xs + j * FK);
                const float4 t1 = *(const float4 *)(xs + j * FK + 4);
#pragma unroll
                for (int rr = 0; rr < R; ++rr) {
                  const float2 xx = make_float2(x[rr][j], x[rr][j]), hh = make_float2(0.5f, 0.5f);   // x = -2 a_j
                  const float2 d0 = __ffma2_rn(xx, hh, make_float2(t0.x, t0.y)), d1 = __ffma2_rn(xx, hh, make_float2(t0.z, t0.w));
                  const float2 d2 = __ffma2_rn(xx, hh, make_float2(t1.x, t1.y)), d3 = __ffma2_rn(xx, hh, make_float2(t1.z, t1.w));
                  r2[rr][0] = __ffma2_rn(d0, d0, r2[rr][0]);
                  r2[rr][1] = __ffma2_rn(d1, d1, r2[rr][1]);
                  r2[rr][2] = __ffma2_rn(d2, d2, r2[rr][2]);
                  r2[rr][3] = __ffma2_rn(d3, d3, r2[rr][3]);
                }
              }
            } else {
              {
                const float4 n0 = *(const float4 *)(xs + (DP + 1) * FK);      // |b_i|^2
                const float4 n1 = *(const float4 *)(xs + (DP + 1) * FK + 4);
#pragma unroll
                for (int rr = 0; rr < R; ++rr) {
                  const float2 aa = make_float2(a2[rr], a2[rr]);
                  r2[rr][0] = __fadd2_rn(aa, make_float2(n0.x, n0.y));
                  r2[rr][1] = __fadd2_rn(aa, make_float2(n0.z, n0.w));
                  r2[rr][2] = __fadd2_rn(aa, make_float2(n1.x, n1.y));
                  r2[rr][3] = __fadd2_rn(aa, make_float2(n1.z, n1.w));
                }
              }
#pragma unroll
              for (int j = 0; j < DP; ++j) {
                const float4 t0 = *(const float4 *)(xs + j * FK);
                const float4 t1 = *(const float4 *)(xs + j * FK + 4);
#pragma unroll
                for (int rr = 0; rr < R; ++rr) {
                  const float2 xx = make_float2(x[rr][j], x[rr][j]);            // -2 a_j
                  r2[rr][0] = __ffma2_rn(xx, make_float2(t0.x, t0.y), r2[rr][0]);
                  r2[rr][1] = __ffma2_rn(xx, make_float2(t0.z, t0.w), r2[rr][1]);
                  r2[rr][2] = __ffma2_rn(xx, make_float2(t1.x, t1.y), r2[rr][2]);
                  r2[rr][3] = __ffma2_rn(xx, make_float2(t1.z, t1.w), r2[rr][3]);
                }
              }
            }
            const float4 al0 = *(const float4 *)(xs + DP * FK);
            const float4 al1 = *(const float4 *)(xs + DP * FK + 4);
            if (rb == 0) mbar_wait_prof(smem_u32(&a_empty[sa]), pa ^ 1, 32, w_aempty, pon);   // stage released by the MMA
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
              float2 kv[4];
              if (matern) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  float2 rad, ex;
                  // |r^2|: rounding can leave -1e-7 where the distance is 0 (MUFU takes the modifier for free)
                  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad.x) : "f"(fabsf(r2[rr][e].x)));
                  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad.y) : "f"(fabsf(r2[rr][e].y)));
                  const float2 arg = __fmul2_rn(rad, make_float2(-3.2259955597f, -3.2259955597f));   // -sqrt5 log2(e)
                  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex.x) : "f"(arg.x));
                  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex.y) : "f"(arg.y));
                  const float2 poly = __ffma2_rn(rad, make_float2(2.2360679775f, 2.2360679775f),
                                                 __ffma2_rn(r2[rr][e], make_float2(1.6666666667f, 1.6666666667f),
                                                            make_float2(1.0f, 1.0f)));
                  kv[e] = __fmul2_rn(poly, ex);
                }
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float2 arg = __fmul2_rn(r2[rr][e], make_float2(-0.7213475204f, -0.7213475204f));  // -0.5 log2(e)
                  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(kv[e].x) : "f"(arg.x));
                  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(kv[e].y) : "f"(arg.y));
                }
              }
              if (do_mu) {
                float2 m2 = __fmul2_rn(kv[0], make_float2(al0.x, al0.y));
                m2 = __ffma2_rn(kv[1], make_float2(al0.z, al0.w), m2);
                m2 = __ffma2_rn(kv[2], make_float2(al1.x, al1.y), m2);
                m2 = __ffma2_rn(kv[3], make_float2(al1.z, al1.w), m2);
                mu_acc[R * rb + rr] += m2.x + m2.y;
              }
              uint32_t hi[4], lo[4];
              if (f16) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  __half2 h = __float22half2_rn(kv[e]);
                  __half2 l = __float22half2_rn(__ffma2_rn(__half22float2(h), make_float2(-1.0f, -1.0f), kv[e]));   // k' - hi, exact
                  hi[e] = *reinterpret_cast<uint32_t *>(&h);
                  lo[e] = *reinterpret_cast<uint32_t *>(&l);
                }
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  __nv_bfloat162 h = __float22bfloat162_rn(kv[e]);
                  const uint32_t hb = *reinterpret_cast<uint32_t *>(&h);
                  const float2 hf = make_float2(__uint_as_float(hb << 16), __uint_as_float(hb & 0xffff0000u));
                  __nv_bfloat162 l = __float22bfloat162_rn(__ffma2_rn(hf, make_float2(-1.0f, -1.0f), kv[e]));
                  hi[e] = hb;
                  lo[e] = *reinterpret_cast<uint32_t *>(&l);
                }
              }
              const int row = lane + 32 * (R * rb + rr);
              const uint32_t off = (uint32_t)((row >> 3) * 1024 + (row & 7) * 128 + (((q ^ (row & 7)) & 7) << 4));
              *(uint4 *)(st_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
              *(uint4 *)(st_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            }
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_u32(&a_full[sa]));
          const uint32_t stage_just_written = smem_u32(sA + sa * STAGE_BYTES);
          if (++sa == NSTA) { sa = 0; pa ^= 1; }
          asm volatile("cp.async.wait_group 0;\n" ::: "memory");          // next slice has landed
          // the previous cache store must have finished READING its stage before anyone overwrites it
          if (store_cache && gt == 0) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
          { long long t0 = pon ? clock64() : 0;
            asm volatile("bar.sync 1, %0;\n" ::"n"(GEN_THREADS));
            if (pon) w_bar += clock64() - t0; }
          if (store_cache && gt == 0) bulk_store(kc + (size_t)kb * STAGE_BYTES, stage_just_written, STAGE_BYTES);
          xbuf ^= 1;
        }
      }
      if (pon && lane == 0) { prm.prof[blockIdx.x * 16 + 5 + 0] = w_aempty; if (q == 0) prm.prof[blockIdx.x * 16 + 6] = w_bar; if (q == 7) prm.prof[blockIdx.x * 16 + 7] = w_bar; }
      // mean: one partial sum per (chunk warp, row)
#pragma unroll
      for (int r4 = 0; r4 < 4; ++r4) mu_sm[q * FM + lane + 32 * r4] = mu_acc[r4];
      asm volatile("bar.sync 1, %0;\n" ::"n"(GEN_THREADS));
      if (gt < FM) {
        const long long cg = tile * FM + gt;
        if (cg < prm.m) {
          float acc = 0.f;
#pragma unroll
          for (int w = 0; w < 8; ++w) acc += mu_sm[w * FM + gt];
          prm.mu_out[cg] = (double)acc;
        }
      }
    }
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512u));
}


// =================================================================================================
// Mean-only pass (the acquisition never reads this model's variance: model 1.. of EHVI / decomposition in the
// reference's semantics, the Pareto-label GP of KEEP).  No tensor core, no operand ring: K1 + the dot product with
// sigma_f2 alpha.  The generator code of the main kernel would leave half of the SM idle here (8 of its 16 warps),
// so this is a separate 256-thread kernel with a few KB of shared memory: two CTAs per SM, 16 K1 warps.
// Warp q owns training points 8q..8q+7 of every 64-block, lane l the candidate rows l + 32 rr, with the main kernel's
// distance form, k' arithmetic and summation order: mu is bit-identical to that of a variance launch.
// =================================================================================================
template <int DP, int R, bool DIRECT>
__global__ void __launch_bounds__(256, 2)
k_posterior_mean_fast(const FastParams prm) {
  constexpr int RB = 128 / (32 * R);
  constexpr int XT_STRIDE = (DP + 2) * FK;
  __shared__ float xc[DP * FM];
  __shared__ __align__(16) float xt[2 * XT_STRIDE];
  __shared__ float mu_sm[8 * FM];
  __shared__ double inv_ell[DP];
  const int tid = threadIdx.x, lane = tid & 31, q = tid >> 5;
  const int d = prm.gp.d, np = prm.gp.n_pad, nkb = np / FK;
  const bool matern = (prm.gp.kernel == OMBO_KERNEL_MATERN52);
  const long long n_tiles = (prm.m + FM - 1) / FM;
  if (tid < DP) inv_ell[tid] = tid < d ? 1.0 / prm.gp.ell[tid] : 0.0;
  constexpr int LD_ROWS = 256 / 16;
  const int ld_j = tid >> 4, ld_o = (tid & 15) * 4;
  constexpr int LD_SWEEPS = (DP + 2 + LD_ROWS - 1) / LD_ROWS;
  auto prefetch_slice = [&](float *dst, int kb) {
#pragma unroll
    for (int sw = 0; sw < LD_SWEEPS; ++sw) {
      const int jj = ld_j + LD_ROWS * sw;
      if (jj <= DP + 1) {
        const float *src = (jj < DP) ? prm.gp.xs32 + (size_t)jj * np + kb * FK + ld_o
                                     : (jj == DP ? prm.gp.alpha32 : prm.gp.b2_32) + kb * FK + ld_o;
        const uint32_t sd = smem_u32(dst + jj * FK + ld_o);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" ::"r"(sd), "l"(src) : "memory");
      }
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
  };
  int xbuf = 0;
  prefetch_slice(xt, 0);
  asm volatile("cp.async.wait_group 0;\n" ::: "memory");
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    __syncthreads();
    for (int e = tid; e < FM * DP; e += 256) {
      const int r_ = e & (FM - 1), j = e >> 7;
      const long long cg = tile * FM + r_;
      xc[j * FM + r_] = (cg < prm.m && j < d)
                            ? -2.0f * (float)((ombo_pool_coord(prm.pool, cg, j) - prm.gp.center[j]) * inv_ell[j])
                            : 0.f;
    }
    __syncthreads();
    float mu_acc[4] = {0.f, 0.f, 0.f, 0.f};
    float x[R][DP], a2[R];
    auto load_rows = [&](int rb) {
#pragma unroll
      for (int rr = 0; rr < R; ++rr) {
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < DP; ++j) { x[rr][j] = xc[j * FM + lane + 32 * (R * rb + rr)]; acc = fmaf(x[rr][j], x[rr][j], acc); }
        a2[rr] = 0.25f * acc;
      }
    };
    if (RB == 1) load_rows(0);
    for (int kb = 0; kb < nkb; ++kb) {
      prefetch_slice(xt + (xbuf ^ 1) * XT_STRIDE, (kb + 1 < nkb) ? kb + 1 : 0);
      const float *xs = xt + xbuf * XT_STRIDE + 8 * q;
#pragma unroll 1
      for (int rb = 0; rb < RB; ++rb) {
        if (RB > 1) {
          // compiler barrier: the training-slice loads below do not depend on rb, and hoisted out of this loop
          // they would hold 8 x DP values per lane (spills at DP = 16 / 24)
          asm volatile("" ::: "memory");
          load_rows(rb);
        }
        float2 r2[R][4];
        if (DIRECT) {
#pragma unroll
          for (int rr = 0; rr < R; ++rr)
#pragma unroll
            for (int e = 0; e < 4; ++e) r2[rr][e] = make_float2(0.f, 0.f);
#pragma unroll
          for (int j = 0; j < DP; ++j) {
            const float4 t0 = *(const float4 *)(xs + j * FK);
            const float4 t1 = *(const float4 *)(xs + j * FK + 4);
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
              const float2 xx = make_float2(x[rr][j], x[rr][j]), hh = make_float2(0.5f, 0.5f);
              const float2 d0 = __ffma2_rn(xx, hh, make_float2(t0.x, t0.y)), d1 = __ffma2_rn(xx, hh, make_float2(t0.z, t0.w));
              const float2 d2 = __ffma2_rn(xx, hh, make_float2(t1.x, t1.y)), d3 = __ffma2_rn(xx, hh, make_float2(t1.z, t1.w));
              r2[rr][0] = __ffma2_rn(d0, d0, r2[rr][0]);
              r2[rr][1] = __ffma2_rn(d1, d1, r2[rr][1]);
              r2[rr][2] = __ffma2_rn(d2, d2, r2[rr][2]);
              r2[rr][3] = __ffma2_rn(d3, d3, r2[rr][3]);
            }
          }
        } else {
          const float4 n0 = *(const float4 *)(xs + (DP + 1) * FK);
          const float4 n1 = *(const float4 *)(xs + (DP + 1) * FK + 4);
#pragma unroll
          for (int rr = 0; rr < R; ++rr) {
            const float2 aa = make_float2(a2[rr], a2[rr]);
            r2[rr][0] = __fadd2_rn(aa, make_float2(n0.x, n0.y));
            r2[rr][1] = __fadd2_rn(aa, make_float2(n0.z, n0.w));
            r2[rr][2] = __fadd2_rn(aa, make_float2(n1.x, n1.y));
            r2[rr][3] = __fadd2_rn(aa, make_float2(n1.z, n1.w));
          }
#pragma unroll
          for (int j = 0; j < DP; ++j) {
            const float4 t0 = *(const float4 *)(xs + j * FK);
            const float4 t1 = *(const float4 *)(xs + j * FK + 4);
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
              const float2 xx = make_float2(x[rr][j], x[rr][j]);
              r2[rr][0] = __ffma2_rn(xx, make_float2(t0.x, t0.y), r2[rr][0]);
              r2[rr][1] = __ffma2_rn(xx, make_float2(t0.z, t0.w), r2[rr][1]);
              r2[rr][2] = __ffma2_rn(xx, make_float2(t1.x, t1.y), r2[rr][2]);
              r2[rr][3] = __ffma2_rn(xx, make_float2(t1.z, t1.w), r2[rr][3]);
            }
          }
        }
        const float4 al0 = *(const float4 *)(xs + DP * FK);
        const float4 al1 = *(const float4 *)(xs + DP * FK + 4);
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
          float2 kv[4];
          if (matern) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float2 rad, ex;
              asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad.x) : "f"(fabsf(r2[rr][e].x)));
              asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad.y) : "f"(fabsf(r2[rr][e].y)));
              const float2 arg = __fmul2_rn(rad, make_float2(-3.2259955597f, -3.2259955597f));
              asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex.x) : "f"(arg.x));
              asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex.y) : "f"(arg.y));
              const float2 poly = __ffma2_rn(rad, make_float2(2.2360679775f, 2.2360679775f),
                                             __ffma2_rn(r2[rr][e], make_float2(1.6666666667f, 1.6666666667f),
                                                        make_float2(1.0f, 1.0f)));
              kv[e] = __fmul2_rn(poly, ex);
            }
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 arg = __fmul2_rn(r2[rr][e], make_float2(-0.7213475204f, -0.7213475204f));
              asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(kv[e].x) : "f"(arg.x));
              asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(kv[e].y) : "f"(arg.y));
            }
          }
          float2 m2 = __fmul2_rn(kv[0], make_float2(al0.x, al0.y));
          m2 = __ffma2_rn(kv[1], make_float2(al0.z, al0.w), m2);
          m2 = __ffma2_rn(kv[2], make_float2(al1.x, al1.y), m2);
          m2 = __ffma2_rn(kv[3], make_float2(al1.z, al1.w), m2);
          const float ms = m2.x + m2.y;
          if (RB == 1 || rb == 0) mu_acc[rr] += ms; else mu_acc[(R + rr) & 3] += ms;
        }
      }
      asm volatile("cp.async.wait_group 0;\n" ::: "memory");
      __syncthreads();
      xbuf ^= 1;
    }
#pragma unroll
    for (int r4 = 0; r4 < 4; ++r4) mu_sm[q * FM + lane + 32 * r4] = mu_acc[r4];
    __syncthreads();
    if (tid < FM) {
      const long long cg = tile * FM + tid;
      if (cg < prm.m) {
        float acc = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) acc += mu_sm[w * FM + tid];
        prm.mu_out[cg] = (double)acc;
        prm.var_out[cg] = nan("");
      }
    }
  }
}

// ---- host side ------------------------------------------------------------------------------
typedef PFN_encodeTiled_t PFN_encodeTiled;

PFN_encodeTiled_t ombo_get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

static int make_b_map(CUtensorMap *map, const void *base, int n_pad, int box_rows, int rows = 0) {
  PFN_encodeTiled enc = ombo_get_encode_tiled();
  if (!enc) { ombo_set_error("cuTensorMapEncodeTiled is not available from the driver"); return OMBO_ERR_CUDA; }
  cuuint64_t dims[2] = {(cuuint64_t)n_pad, (cuuint64_t)(rows ? rows : n_pad)};
  cuuint64_t strides[1] = {(cuuint64_t)n_pad * 2};
  cuuint32_t box[2] = {FK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { ombo_set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return OMBO_ERR_CUDA; }
  return OMBO_OK;
}

// the K* cache seen as rows of 128 B (one shared-memory stage = 256 rows), no swizzle: a straight copy
int ombo_make_linear_map(CUtensorMap *map, const void *base, size_t rows) {
  PFN_encodeTiled enc = ombo_get_encode_tiled();
  if (!enc) { ombo_set_error("cuTensorMapEncodeTiled is not available from the driver"); return OMBO_ERR_CUDA; }
  cuuint64_t dims[2] = {64, (cuuint64_t)rows};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {64, 256};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { ombo_set_error("cuTensorMapEncodeTiled (cache) failed (%d)", (int)r); return OMBO_ERR_CUDA; }
  return OMBO_OK;
}

int ombo_fast_path_built() { return 1; }

template <int DP, int R, bool F16>
static int launch_fast(ombo_ctx *ctx, const CUtensorMap &map_hi, const CUtensorMap &map_lo, const CUtensorMap &map_kc, const FastParams &prm,
                       int grid, cudaStream_t s) {
  const size_t smem = (size_t)6 * STAGE_BYTES + (size_t)DP * FM * 4 + 2 * (size_t)(DP + 2) * FK * 4 +
                      8 * FM * 4 + 16 + 24 * 8 + 24 * 8 + 1024;   // barriers + TMEM slot, 1/lengthscale, alignment slack
  // set on every launch: the attribute belongs to the (function, device) pair, and one process may drive several devices
  OMBO_CUDA(cudaFuncSetAttribute(k_posterior_fast<DP, R, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ProfScope prof(ctx, s);
  k_posterior_fast<DP, R, F16><<<grid, 16 * 32, smem, s>>>(map_hi, map_lo, map_kc, prm);
  return OMBO_OK;
}

int ombo_posterior_fast(ombo_ctx *ctx, const GpDev &gp, const PoolDev &pool, long long m, double *mu, double *var,
                        bool want_var, cudaStream_t s, const FuseAcq *fuse_req, int *fused, int bound_chunks) {
  if (fused) *fused = 0;
  if (m <= 0) return OMBO_OK;
  if (gp.d > 24) {
    ombo_set_error("fast precision mode supports d <= 24 (got %d); use OMBO_PREC_FP64", gp.d);
    return OMBO_ERR_UNSUPPORTED;
  }
  long long tiles = (m + FM - 1) / FM;
  const ombo_knobs &kn = ctx->knobs;
  if (!want_var) {
    // mean-only: the dedicated K1 kernel (two CTAs per SM; rows per lane and dimension padding as in the main kernel)
    FastParams prm = {};
    prm.gp = gp; prm.pool = pool; prm.m = m; prm.mu_out = mu; prm.var_out = var;
    const int grid = (int)(tiles < 2LL * ctx->num_sms ? tiles : 2LL * ctx->num_sms);
    const bool direct = (gp.flags & OMBO_GP_FP16_PLANES) != 0;
    ProfScope prof(ctx, s);
#define MEAN_CASE(DPV, RV)                                                                              \
    if (gp.d <= DPV) {                                                                                  \
      if (direct) k_posterior_mean_fast<DPV, RV, true><<<grid, 256, 0, s>>>(prm);                       \
      else k_posterior_mean_fast<DPV, RV, false><<<grid, 256, 0, s>>>(prm);                             \
    } else
    MEAN_CASE(2, 4) MEAN_CASE(4, 4) MEAN_CASE(6, 4) MEAN_CASE(8, 4) MEAN_CASE(10, 4) MEAN_CASE(12, 4) MEAN_CASE(16, 2)
    { if (direct) k_posterior_mean_fast<24, 2, true><<<grid, 256, 0, s>>>(prm);
      else k_posterior_mean_fast<24, 2, false><<<grid, 256, 0, s>>>(prm); }
#undef MEAN_CASE
    ctx->launches += 1;
    OMBO_CUDA(cudaGetLastError());
    return OMBO_OK;
  }
  if (gp.flags & OMBO_GP_F8C_PLANES) return ombo_posterior_fast8(ctx, gp, pool, m, mu, var, s, fuse_req, fused, bound_chunks);
  CUtensorMap map_hi, map_lo, map_kc;
  int rc = make_b_map(&map_hi, gp.bhi, gp.n_pad, 256);
  if (rc) return rc;
  rc = make_b_map(&map_lo, gp.blo, gp.n_pad, 256);
  if (rc) return rc;
  FastParams prm = {};
  prm.gp = gp; prm.pool = pool; prm.m = m; prm.mu_out = mu; prm.var_out = var;
  const bool want_prof = kn.fast_profile != 0;
  if (want_prof && !ctx->prof_dev) OMBO_CUDA(cudaMalloc(&ctx->prof_dev, 16 * 256 * sizeof(long long)));
  long long *prof_dev = ctx->prof_dev;
  prm.prof = want_prof ? prof_dev : nullptr;
  if (want_prof) OMBO_CUDA(cudaMemsetAsync(prof_dev, 0, 16 * 256 * sizeof(long long), s));
  const int grid = (int)(tiles < ctx->num_sms ? tiles : ctx->num_sms);
  // the two planes are adjacent in the state blob (gp_layout): one map of 64-row boxes over (2 n_pad, n_pad) serves both
  rc = make_b_map(&map_kc, gp.bhi, gp.n_pad, 64, 2 * gp.n_pad);
  if (rc) return rc;
  if (gp.n_pad > 512) {            // more than one TMEM pass: generated K* blocks are cached in L2
    rc = ombo_ws_reserve(&ctx->ws_scratch, &ctx->ws_scratch_bytes, (size_t)grid * (gp.n_pad / FK) * STAGE_BYTES);
    if (rc) return rc;
    prm.kcache = (unsigned char *)ctx->ws_scratch;
  }
  const int d = gp.d;
  // (16 generator warps with 2 rows per lane were measured too: the same number of independent chains per
  // scheduler, no gain -- the instantiations were dropped to keep the build short)
  const bool f16 = (gp.flags & OMBO_GP_FP16_PLANES) != 0;     // format of the planes, as reported by the refresh
#define FAST_DISPATCH(DPV, RV)                                                                                \
  rc = f16 ? launch_fast<DPV, RV, true>(ctx, map_hi, map_lo, map_kc, prm, grid, s)                            \
           : launch_fast<DPV, RV, false>(ctx, map_hi, map_lo, map_kc, prm, grid, s)
  if (d <= 2) { FAST_DISPATCH(2, 4); }
  else if (d <= 4) { FAST_DISPATCH(4, 4); }
  else if (d <= 6) { FAST_DISPATCH(6, 4); }
  else if (d <= 8) { FAST_DISPATCH(8, 4); }
  else if (d <= 10) { FAST_DISPATCH(10, 4); }
  else if (d <= 12) { FAST_DISPATCH(12, 4); }
  else if (d <= 16) { FAST_DISPATCH(16, 2); }
  else { FAST_DISPATCH(24, 2); }
#undef FAST_DISPATCH
  if (rc) return rc;
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  if (want_prof) {
    static long long h[16 * 256];
    OMBO_CUDA(cudaStreamSynchronize(s));
    OMBO_CUDA(cudaMemcpy(h, prof_dev, sizeof(h), cudaMemcpyDeviceToHost));
    double a[8] = {0};
    for (int b = 0; b < grid; ++b) for (int k = 0; k < 8; ++k) a[k] += (double)h[b * 16 + k] / grid;
    fprintf(stderr, "[fast prof] per-CTA cycles: tma.wait_b_empty %.0f / tma.total %.0f | mma.wait_a_full %.0f wait_b_full %.0f "
            "wait_t_empty %.0f | gen.wait_a_empty %.0f gen.bar(w0) %.0f gen.bar(w7) %.0f  (tiles/CTA %.1f)\n",
            a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], (double)tiles / grid);
  }
  return OMBO_OK;
}
