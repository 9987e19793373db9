// Stage 1 of the pruned arg-max (api.cu, score_pruned) with the distances on the tensor core: the mean-only upper bound
// of the exact 2-D EHVI for both GPs of an f8c pair, like k_posterior_mean8, but with a certified margin on the mean
// instead of the full launch's bits.
//
//   r~^2 = x_lo.b_hi + x_hi.b_lo + x_hi.b_hi + (a2_hi + a2_lo + b2_hi + b2_lo)   (tcgen05.mma kind::f16, FP32 in TMEM)
//   mu~  = sum_i c_i k'(r~_i^2),  A = sum_i |c_i| k'(r~_i^2)          (c = sigma_f2 alpha; consumers, FP32)
//   UB   = ehvi2d_value<float>(mu~0 - M0, mu~1 - M1, var0_up, var1_up)  with M >= |mu~ - mu_F| (DESIGN.md section 4)
//
// x is the full launch's FP32 candidate coordinate (gen8_coord) and b its FP32 training coordinate, each split into
// fp16 hi + lo parts; |b|^2 and a2 = |x|^2 / 4 ride in K columns 12..15 of the hi planes, so TMEM holds r^2 itself.
// A row of either operand is 128 B: [GP 0 hi | GP 0 lo | GP 1 hi | GP 1 lo], 16 fp16 each (d <= 12), SWIZZLE_128B.
// Both GPs' training planes and c, |c| stay in shared memory for the whole launch (n_pad 1024: 144 KB).
//
// One persistent CTA per SM, 128 candidates per tile, TMEM as two 256-column accumulator slots; no CTA barrier after
// the prologue, every hand-off an mbarrier:
//   warps 0..15   consumers: warp w reads TMEM lanes 32 (w & 3).. (its rows) and a quarter of each chunk's columns
//                 (group w >> 2), evaluates k' (sqrt on MUFU; ex2 on MUFU or, for S1_POLY_* of every 16 column
//                 pairs, as a polynomial on the FMA pipe) and accumulates mu~ and A per GP; per tile the partials go
//                 to a double-buffered table in shared memory
//   warps 16..19  producers / bound: thread r builds row r of the A tile of tile t (pool coordinate, FP64 prep, fp16
//                 split), then finishes tile t - 1: the four partials, the margin, the EHVI bound and the per-CTA best
//   warp 20       MMA issuer: per 256-column chunk three tcgen05.mma (the two lo products first, from 0, then hi.hi)
#include <algorithm>

#include "acq_math.cuh"
#include "gen8.cuh"
#include "umma.cuh"

#define S1_ROWS 128
#define S1_CW 256                          // accumulator slot width (TMEM 512 columns = 2 slots)
#define S1_CONS 16                         // consumer warps: 4 column groups x 4 TMEM lane quarters
#define S1_PROD 4                          // producer / bound warps: one thread per candidate row
#define S1_MMA_WARP (S1_CONS + S1_PROD)
#define S1_THREADS ((S1_MMA_WARP + 1) * 32)
#define S1_TILE_BYTES (S1_ROWS * 128)
// column pairs out of every 16 whose ex2 runs as a polynomial on the FMA pipe (the rest on MUFU).  Matern: timed on the
// C5 headline at 0 / 2 / 4 / 8 / 12 / 16 (DESIGN.md section 4), 4 is the fastest; RBF: 4, not timed
#ifndef S1_POLY_MATERN
#define S1_POLY_MATERN 4
#endif
#ifndef S1_POLY_RBF
#define S1_POLY_RBF 4
#endif

// ---- the margin (DESIGN.md section 4, "Stage 1 on the tensor core"); units of u = 2^-24 ----
#define S1_U 5.9604644775390625e-8
#define S1_G_F 13.0        // full launch's FP32 r^2 chain: one add + up to 12 FMAs, each <= u T
#define S1_G_TC 56.0       // fp16 hi/lo split (3 x 4 u on the products, 4 u on the norms) + the MMA's FP32 sums (40 u)
#define S1_E_SUB (14.0 * 0.5 * S1_U)   // fp16 subnormal parts: 2^-25 (d + 2)
#define S1_ETA (48.0 * S1_U)           // relative error of k' evaluated from r^2, both paths
#define S1_ETA_ABS (32.0 * S1_U)       // the rounding of r (and of the ex2 argument) weighted by |dk/dr| r <= 2, times S
#define S1_SAFETY 4.0
#define S1_ER_MAX 0.0078125            // beyond this r^2 error the bound is not formed (UB = NaN: the candidate survives)
// the launch gate (ombo_stage1_tc_useful): the tensor-core stage 1 runs only while M / A stays below this for the
// pool's largest T; above it the exact-mean stage 1 keeps fewer survivors at no larger cost (DESIGN.md section 4)
#define S1_REL_MAX 1e-3

// the margin relative to A = sum |c| k' for a candidate with T = (sqrt(a2) + sqrt(max |b|^2))^2, and the r^2 error
// e_r it rests on: M = s1_rel_margin(T) A + S1_SAFETY S1_ETA_ABS S.  Matern: 5/6 (k' of r) plus 10/3 e_f (the full
// launch's signed 5/3 r^2 where its r^2 < 0); RBF: 1/2.  The factors 1.05 / 1.02 take k' at the intermediate point
// back to k'(r~^2) and hold while e_r <= S1_ER_MAX.
__host__ __device__ inline double s1_rel_margin(double T, bool matern, int n_pad, double &e_r) {
  const double e_f = S1_G_F * S1_U * T;
  e_r = (S1_G_F + S1_G_TC) * S1_U * T + S1_E_SUB;
  const double lr = matern ? (5.0 / 6.0) * 1.05 * e_r + (10.0 / 3.0) * 1.02 * e_f : 0.5 * 1.05 * e_r;
  const double zeta = (3.0 * n_pad / 64.0 + 16.0) * S1_U;            // summation of both means
  return S1_SAFETY * (lr + S1_ETA + zeta) * 1.05;
}

// 2^t for t <= 0 on the FMA pipe: n = rint(t) by the 1.5 * 2^23 shift, f = t - n in [-0.5, 0.5] (exact), a degree-5
// polynomial for 2^f (relative error 1.6e-7 in exact arithmetic, <= 2^-21 in FP32: tests/test_prune_stage1_tc_cpu.py
// checks every FP32 f with |f| >= 2^-12 and a dense sample below), and n added to the exponent field.  t is clamped
// at -125, where the result is still normal; ex2.approx.ftz flushes below 2^-126, so the two differ by less than
// 2^-124 there.
__device__ __forceinline__ float2 s1_exp2_poly(float2 t) {
  t.x = fmaxf(t.x, -125.f);
  t.y = fmaxf(t.y, -125.f);
  const float2 sh = make_float2(12582912.f, 12582912.f);
  const float2 j = __fadd2_rn(t, sh);
  const float2 n = __fadd2_rn(j, make_float2(-12582912.f, -12582912.f));
  const float2 f = __ffma2_rn(n, make_float2(-1.f, -1.f), t);
  float2 p = make_float2(1.3276718091219664e-3f, 1.3276718091219664e-3f);
  p = __ffma2_rn(p, f, make_float2(9.675543755292892e-3f, 9.675543755292892e-3f));
  p = __ffma2_rn(p, f, make_float2(5.5507123470306396e-2f, 5.5507123470306396e-2f));
  p = __ffma2_rn(p, f, make_float2(2.4022120237350464e-1f, 2.4022120237350464e-1f));
  p = __ffma2_rn(p, f, make_float2(6.931469440460205e-1f, 6.931469440460205e-1f));
  p = __ffma2_rn(p, f, make_float2(1.0000001192092896f, 1.0000001192092896f));
  return make_float2(__uint_as_float(__float_as_uint(p.x) + (__float_as_uint(j.x) << 23)),
                     __uint_as_float(__float_as_uint(p.y) + (__float_as_uint(j.y) << 23)));
}

struct Stage1Gp {
  const float *xs32, *alpha32, *b2_32;
  const double *ell, *center;
  int n_pad;
  float var_up;
  int matern;
};

struct Stage1Params {
  Stage1Gp gp[2];
  PoolDev pool;
  long long m;
  int d, n_pf, nb;                    // nb: rows of the B planes, max n_pad
  float c00, c01;
  const double *stripes;
  double *ub;                         // [m]
  double *mu_out, *marg_out;          // optional [2][m] each: mu~ and M as doubles (tests)
  ombo_best *partials;                // [gridDim.x]
};

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t *v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

// 16 accumulator columns of one row: k' and the sums (mu~, A), two columns per packed operation; cq: per column pair
// {c0, c1, |c0|, |c1|}.  e0: the pair index within the 16 pairs of 32 columns (the polynomial share)
template <bool MATERN, int E0>
__device__ __forceinline__ void s1_columns(const uint32_t (&v)[16], const float4 *cq, float2 (&mu)[2], float2 (&ab)[2]) {
  constexpr int NPOLY = MATERN ? S1_POLY_MATERN : S1_POLY_RBF;
#pragma unroll
  for (int ee = 0; ee < 8; ++ee) {
    const int e = E0 + ee;
    const float2 r2 = make_float2(__uint_as_float(v[2 * ee]), __uint_as_float(v[2 * ee + 1]));
    float2 kv;
    if (MATERN) {
      // k' = (1 + sqrt5 r + 5/3 r^2) e^(-sqrt5 r) with r = sqrt|r~^2|: the Matern function of r, 5/6-Lipschitz in r^2
      // relative to k' (the full launch's 5/3 r^2 term takes the signed r^2; DESIGN.md section 4)
      float2 rad, ex;
      asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad.x) : "f"(fabsf(r2.x)));
      asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad.y) : "f"(fabsf(r2.y)));
      const float2 arg = __fmul2_rn(rad, make_float2(-3.2259955597f, -3.2259955597f));   // -sqrt5 log2(e)
      if (e < NPOLY) {
        ex = s1_exp2_poly(arg);
      } else {
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex.x) : "f"(arg.x));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex.y) : "f"(arg.y));
      }
      const float2 t = __ffma2_rn(rad, make_float2(1.6666666667f, 1.6666666667f), make_float2(2.2360679775f, 2.2360679775f));
      kv = __fmul2_rn(__ffma2_rn(rad, t, make_float2(1.f, 1.f)), ex);
    } else {
      const float2 arg = __fmul2_rn(r2, make_float2(-0.7213475204f, -0.7213475204f));     // -0.5 log2(e)
      if (e < NPOLY) {
        kv = s1_exp2_poly(arg);
      } else {
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(kv.x) : "f"(arg.x));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(kv.y) : "f"(arg.y));
      }
    }
    const float4 c = cq[ee];
    mu[e & 1] = __ffma2_rn(kv, make_float2(c.x, c.y), mu[e & 1]);
    ab[e & 1] = __ffma2_rn(kv, make_float2(c.z, c.w), ab[e & 1]);
  }
}

// one consumer group's columns of a chunk (32 or 64), 16 TMEM columns per load, the next load in flight while the
// current 16 columns are evaluated
template <bool MATERN>
__device__ __forceinline__ void s1_group(uint32_t taddr, int ncols, const float4 *cq, float2 (&acc)[4]) {
  float2 mu[2] = {acc[0], acc[1]}, ab[2] = {acc[2], acc[3]};
  uint32_t va[16], vb[16];
  tmem_ld16(taddr, va);
  tmem_ld_wait();
  for (int l = 0; l < ncols; l += 32) {
    tmem_ld16(taddr + (uint32_t)(l + 16), vb);
    s1_columns<MATERN, 0>(va, cq + l / 2, mu, ab);
    tmem_ld_wait();
    if (l + 32 < ncols) tmem_ld16(taddr + (uint32_t)(l + 32), va);
    s1_columns<MATERN, 8>(vb, cq + l / 2 + 8, mu, ab);
    tmem_ld_wait();
  }
  acc[0] = mu[0]; acc[1] = mu[1]; acc[2] = ab[0]; acc[3] = ab[1];
}

// chunk k of a tile: GP g and its first training column
__device__ __forceinline__ void s1_chunk(const Stage1Params &p, int k, int &g, int &col0, int &n) {
  const int nc0 = (p.gp[0].n_pad + S1_CW - 1) / S1_CW;
  g = k < nc0 ? 0 : 1;
  col0 = (g ? k - nc0 : k) * S1_CW;
  n = min(S1_CW, p.gp[g].n_pad - col0);
}

__device__ __forceinline__ uint32_t s1_pack(float lo, float hi) {
  return (uint32_t)__half_as_ushort(__float2half_rn(lo)) | ((uint32_t)__half_as_ushort(__float2half_rn(hi)) << 16);
}

// one 16-byte chunk (8 fp16) of a 128-B operand row in the SWIZZLE_128B layout
__device__ __forceinline__ void s1_store_chunk(unsigned char *base, int row, int ch, const float (&v)[8]) {
  const uint32_t off = (uint32_t)((row >> 3) * 1024 + (row & 7) * 128 + (((ch ^ (row & 7)) & 7) << 4));
  *(uint4 *)(base + off) = make_uint4(s1_pack(v[0], v[1]), s1_pack(v[2], v[3]), s1_pack(v[4], v[5]), s1_pack(v[6], v[7]));
}

// the 16 K columns of one GP of one operand row, hi and lo plane: coordinates 0..11, then the norm columns
// (A: [a2_hi, a2_lo, 1, 1], B: [1, 1, b2_hi, b2_lo]; zero in the lo planes)
__device__ __forceinline__ void s1_split_row(const float (&x)[12], float nrm, bool is_a, float (&hi)[16], float (&lo)[16]) {
#pragma unroll
  for (int j = 0; j < 12; ++j) {
    const float h = __half2float(__float2half_rn(x[j]));
    hi[j] = h;
    lo[j] = x[j] - h;
  }
  const float nh = __half2float(__float2half_rn(nrm)), nl = nrm - nh;
  hi[12] = is_a ? nh : 1.f; hi[13] = is_a ? nl : 1.f; hi[14] = is_a ? 1.f : nh; hi[15] = is_a ? 1.f : nl;
#pragma unroll
  for (int j = 12; j < 16; ++j) lo[j] = 0.f;
}

__device__ __forceinline__ void s1_store_gp(unsigned char *base, int row, int g, const float (&hi)[16], const float (&lo)[16]) {
  float t[8];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
#pragma unroll
    for (int j = 0; j < 8; ++j) t[j] = hi[8 * h + j];
    s1_store_chunk(base, row, 4 * g + h, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) t[j] = lo[8 * h + j];
    s1_store_chunk(base, row, 4 * g + 2 + h, t);
  }
}

// fp16 range: every coordinate and norm below 2^15, so hi and lo parts are finite (margin to 65504)
__device__ __forceinline__ bool s1_in_range(const float (&x)[12], float nrm) {
  bool ok = nrm < 32768.f;
#pragma unroll
  for (int j = 0; j < 12; ++j) ok = ok && fabsf(x[j]) < 32768.f;
  return ok;
}

template <bool MAT0, bool MAT1>
__global__ void __launch_bounds__(S1_THREADS, 1) k_stage1_tc(const __grid_constant__ Stage1Params p) {
  extern __shared__ __align__(1024) unsigned char s1_smem[];
  unsigned char *sB = s1_smem + ((1024u - (smem_u32(s1_smem) & 1023u)) & 1023u);
  unsigned char *sA = sB + (size_t)p.nb * 128;                      // 2 tiles
  float4 *cq = (float4 *)(sA + 2 * S1_TILE_BYTES);                 // [2][nb / 2] {c0, c1, |c0|, |c1|} per column pair
  float *part = (float *)(cq + p.nb);                                      // [2 buf][4 groups][4: mu0, A0, mu1, A1][128]
  float *ystr = part + 2 * 4 * 4 * S1_ROWS;
  double *geo = (double *)(((uintptr_t)(ystr + 2 * (p.n_pf + 2)) + 15) & ~(uintptr_t)15);   // [2][centre 12, 1/ell 12]
  double *red_v = geo + 48;
  long long *red_i = (long long *)(red_v + S1_PROD);
  float *gpc = (float *)(red_i + S1_PROD);                          // [2][b2 max, S]
  uint64_t *bars = (uint64_t *)(((uintptr_t)(gpc + 4) + 15) & ~(uintptr_t)15);
  uint64_t *a_full = bars, *a_empty = bars + 2, *t_full = bars + 4, *t_empty = bars + 6, *p_full = bars + 8,
           *p_empty = bars + 10;
  uint32_t *tmem_slot = (uint32_t *)(bars + 12);
  int *bad = (int *)(tmem_slot + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&a_full[i]), S1_PROD);
      mbar_init(smem_u32(&a_empty[i]), 1);
      mbar_init(smem_u32(&t_full[i]), 1);
      mbar_init(smem_u32(&t_empty[i]), S1_CONS);
      mbar_init(smem_u32(&p_full[i]), S1_CONS);
      mbar_init(smem_u32(&p_empty[i]), S1_PROD * 32);
    }
    fence_mbar_init();
    for (int i = 0; i < 4; ++i) gpc[i] = 0.f;
    *bad = 0;
  }
  if (warp == S1_MMA_WARP) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::);
  }
  if (tid < 24) {
    const int gi = tid / 12, j = tid % 12;
    geo[gi * 24 + j] = j < p.d ? p.gp[gi].center[j] : 0.0;
    geo[gi * 24 + 12 + j] = j < p.d ? 1.0 / p.gp[gi].ell[j] : 0.0;
  }
  for (int i = tid; i < 2 * (p.n_pf + 2); i += S1_THREADS) ystr[i] = (float)p.stripes[i];
  __syncthreads();
  // training planes of both GPs (one thread per (point, GP)), c and |c|, max |b|^2 and S = sum |c| per GP
  for (int e = tid; e < 2 * p.nb; e += S1_THREADS) {
    const int g = e / p.nb, i = e % p.nb;
    const Stage1Gp &G = p.gp[g];
    float x[12], nrm = 0.f, c = 0.f;
#pragma unroll
    for (int j = 0; j < 12; ++j) x[j] = 0.f;
    if (i < G.n_pad) {
#pragma unroll
      for (int j = 0; j < 12; ++j)
        if (j < p.d) x[j] = G.xs32[(size_t)j * G.n_pad + i];
      nrm = G.b2_32[i];
      c = G.alpha32[i];
    }
    if (!s1_in_range(x, nrm)) atomicExch(bad, 1);
    float hi[16], lo[16];
    s1_split_row(x, nrm, false, hi, lo);
    s1_store_gp(sB, i, g, hi, lo);
    float *cp = (float *)(cq + (g * p.nb + i) / 2) + (i & 1);
    cp[0] = c;
    cp[2] = fabsf(c);
    atomicMax((int *)&gpc[2 * g], __float_as_int(nrm));                // nrm >= 0: int order is float order
  }
  __syncthreads();
  if (warp < 2) {                                                   // S = sum |c| of GP `warp`, in a fixed order
    float sum = 0.f;
    for (int i = lane; i < p.nb; i += 32) sum += ((const float *)(cq + (warp * p.nb + i) / 2))[2 + (i & 1)];
#pragma unroll
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) gpc[2 * warp + 1] = sum;
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const long long n_tiles = (p.m + S1_ROWS - 1) / S1_ROWS;
  const int n_iter = (int)((n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);
  const int n_chunks = (p.gp[0].n_pad + S1_CW - 1) / S1_CW + (p.gp[1].n_pad + S1_CW - 1) / S1_CW;

  if (warp == S1_MMA_WARP) {
    // =============================== MMA issuer ===============================
    if (elect_one()) {
      int kc = 0;                                                   // chunks issued so far (slot kc & 1)
      for (int it = 0; it < n_iter; ++it) {
        const int ab = it & 1;
        mbar_wait_sleep(smem_u32(&a_full[ab]), (it >> 1) & 1, MMA_SLEEP_NS);
        tc_fence_after();
        const uint32_t a0 = smem_u32(sA + ab * S1_TILE_BYTES);
        for (int k = 0; k < n_chunks; ++k, ++kc) {
          int g, col0, n;
          s1_chunk(p, k, g, col0, n);
          const int slot = kc & 1;
          mbar_wait_sleep(smem_u32(&t_empty[slot]), ((kc >> 1) & 1) ^ 1, MMA_SLEEP_NS);
          tc_fence_after();
          const uint32_t dst = tmem_base + (uint32_t)(slot * S1_CW);
          const uint32_t idesc = (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(S1_ROWS >> 4) << 24);  // f16 x f16 -> f32
          const uint32_t ah = a0 + 64 * g, bh = smem_u32(sB) + (uint32_t)col0 * 128 + 64 * g;
          // the lo products first, from zero: the hi.hi product (with the norms) then rounds against a small sum
          umma_bf16(dst, make_sdesc(ah + 32), make_sdesc(bh), idesc, 0u);
          umma_bf16(dst, make_sdesc(ah), make_sdesc(bh + 32), idesc, 1u);
          umma_bf16(dst, make_sdesc(ah), make_sdesc(bh), idesc, 1u);
          umma_commit(smem_u32(&t_full[slot]));
        }
        umma_commit(smem_u32(&a_empty[ab]));
      }
    }
  } else if (warp < S1_CONS) {
    // =============================== consumers ================================
    const int q = warp & 3, grp = warp >> 2, row = 32 * q + lane;
    int kc = 0;
    for (int it = 0; it < n_iter; ++it) {
      float2 acc0[4], acc1[4];                                      // per GP: mu (2 chains), A (2 chains)
#pragma unroll
      for (int u = 0; u < 4; ++u) { acc0[u] = make_float2(0.f, 0.f); acc1[u] = make_float2(0.f, 0.f); }
      for (int k = 0; k < n_chunks; ++k, ++kc) {
        int g, col0, n;
        s1_chunk(p, k, g, col0, n);
        const int slot = kc & 1;
        mbar_wait_sleep(smem_u32(&t_full[slot]), (kc >> 1) & 1, 64);
        tc_fence_after();
        const int c = grp * (n >> 2);                               // this group's columns: a quarter of the chunk
        const uint32_t taddr = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(slot * S1_CW + c);
        const float4 *cq_ = cq + (g * p.nb + col0 + c) / 2;
        if (g == 0) s1_group<MAT0>(taddr, n >> 2, cq_, acc0);
        else s1_group<MAT1>(taddr, n >> 2, cq_, acc1);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&t_empty[slot]));
      }
      const int pb = it & 1;
      mbar_wait_sleep(smem_u32(&p_empty[pb]), ((it >> 1) & 1) ^ 1, 64);
      float *pt = part + (size_t)(pb * 4 + grp) * 4 * S1_ROWS;
      pt[0 * S1_ROWS + row] = (acc0[0].x + acc0[0].y) + (acc0[1].x + acc0[1].y);
      pt[1 * S1_ROWS + row] = (acc0[2].x + acc0[2].y) + (acc0[3].x + acc0[3].y);
      pt[2 * S1_ROWS + row] = (acc1[0].x + acc1[0].y) + (acc1[1].x + acc1[1].y);
      pt[3 * S1_ROWS + row] = (acc1[2].x + acc1[2].y) + (acc1[3].x + acc1[3].y);
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&p_full[pb]));
    }
  } else {
    // =============================== producers / bound ========================
    const int r = tid - S1_CONS * 32;                               // candidate row 0..127
    const bool bad_b = *bad != 0;
    BestPair best;
    best.v = -INFINITY; best.i = 0x7fffffffffffffffLL;
    float a2p[2] = {0.f, 0.f};
    bool okp = false;
    auto bound = [&](int t) {
      const long long tile = blockIdx.x + (long long)t * gridDim.x, cg = tile * S1_ROWS + r;
      const int pb = t & 1;
      mbar_wait_sleep(smem_u32(&p_full[pb]), (t >> 1) & 1, 64);
      float mu[2], A[2];
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        const float *pt = part + (size_t)pb * 4 * 4 * S1_ROWS;
        float s = 0.f, a = 0.f;
#pragma unroll
        for (int gr = 0; gr < 4; ++gr) {
          s += pt[(gr * 4 + 2 * g) * S1_ROWS + r];
          a += pt[(gr * 4 + 2 * g + 1) * S1_ROWS + r];
        }
        mu[g] = s; A[g] = a;
      }
      mbar_arrive(smem_u32(&p_empty[pb]));
      if (cg >= p.m) return;
      float lo[2], marg[2];
      bool ok = okp;
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        const bool mat = g == 0 ? MAT0 : MAT1;
        const double sa = sqrt((double)a2p[g]) + sqrt((double)gpc[2 * g]);
        const double T = sa * sa;                                   // >= |b|^2 + a2 + sum |x_j b_j| for every column
        double e_r;
        const double rel = s1_rel_margin(T, mat, p.gp[g].n_pad, e_r);
        ok = ok && e_r <= S1_ER_MAX;
        const double M = rel * (double)A[g] + S1_SAFETY * S1_ETA_ABS * (double)gpc[2 * g + 1];
        marg[g] = (float)M;
        lo[g] = __fsub_rd(mu[g], __double2float_ru(M));
      }
      float ubv;
      if (ok) {
        const int P = p.n_pf;
        ubv = ehvi2d_value<float>(lo[0], lo[1], p.gp[0].var_up, p.gp[1].var_up, ystr, ystr + (P + 2), P, true, p.c00,
                                  p.c01);
      } else {
        ubv = __int_as_float(0x7fffffff);
      }
      p.ub[cg] = (double)ubv;
      if (p.mu_out) {
        p.mu_out[cg] = (double)mu[0]; p.mu_out[p.m + cg] = (double)mu[1];
        p.marg_out[cg] = (double)marg[0]; p.marg_out[p.m + cg] = (double)marg[1];
      }
      const double val = isnan(ubv) ? -INFINITY : (double)ubv;
      const long long gi = p.pool.index_base + cg;
      if (better(val, gi, best.v, best.i)) { best.v = val; best.i = gi; }
    };
    for (int it = 0; it < n_iter; ++it) {
      const int ab = it & 1;
      const long long tile = blockIdx.x + (long long)it * gridDim.x, cg = tile * S1_ROWS + r;
      float x[2][12], a2[2];
#pragma unroll
      for (int g = 0; g < 2; ++g)
#pragma unroll
        for (int j = 0; j < 12; ++j) x[g][j] = 0.f;
      if (cg < p.m) {
#pragma unroll
        for (int j = 0; j < 12; ++j) {
          if (j >= p.d) break;
          const double a = ombo_pool_coord(p.pool, cg, j);
          x[0][j] = gen8_coord(a, geo[j], geo[12 + j]);
          x[1][j] = gen8_coord(a, geo[24 + j], geo[36 + j]);
        }
      }
      bool ok = !bad_b;
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        float s = 0.f;                                              // a2 as gen8_load_row forms it
#pragma unroll
        for (int j = 0; j < 12; ++j) s = fmaf(x[g][j], x[g][j], s);
        a2[g] = 0.25f * s;
        ok = ok && s1_in_range(x[g], a2[g]);
      }
      mbar_wait_sleep(smem_u32(&a_empty[ab]), ((it >> 1) & 1) ^ 1, 64);
      unsigned char *tA = sA + ab * S1_TILE_BYTES;
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        float hi[16], lo[16];
        s1_split_row(x[g], a2[g], true, hi, lo);
        s1_store_gp(tA, r, g, hi, lo);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&a_full[ab]));
      if (it > 0) bound(it - 1);
      a2p[0] = a2[0]; a2p[1] = a2[1]; okp = ok;
    }
    if (n_iter > 0) bound(n_iter - 1);
    best = warp_best(best);
    if (lane == 0) { red_v[warp - S1_CONS] = best.v; red_i[warp - S1_CONS] = best.i; }
  }

  tc_fence_before();
  __syncthreads();
  if (tid == 0) {
    BestPair b;
    b.v = red_v[0]; b.i = red_i[0];
    for (int w = 1; w < S1_PROD; ++w)
      if (better(red_v[w], red_i[w], b.v, b.i)) { b.v = red_v[w]; b.i = red_i[w]; }
    p.partials[blockIdx.x].value = b.v;
    p.partials[blockIdx.x].index = b.i;
  }
  if (warp == S1_MMA_WARP) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512u));
  }
}

// the largest a2 = sum_j ((a_j - c_j) / ell_j)^2 of the pool and max |b|^2, per GP, as double bits into ext[4]
// (zero-initialised; non-negative doubles order as their bits): a counter pool from its box, an explicit one by a scan
__global__ void k_stage1_extent(Stage1Gp g0, Stage1Gp g1, PoolDev pool, long long m, int d, unsigned long long *ext) {
  const Stage1Gp *G[2] = {&g0, &g1};
  double a2[2] = {0.0, 0.0}, b2[2] = {0.0, 0.0};
  const long long stride = (long long)gridDim.x * blockDim.x, t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (int g = 0; g < 2; ++g)
    for (long long i = t0; i < G[g]->n_pad; i += stride) b2[g] = fmax(b2[g], (double)G[g]->b2_32[i]);
  if (pool.X == nullptr) {
    if (t0 == 0)
      for (int g = 0; g < 2; ++g)
        for (int j = 0; j < d; ++j) {
          const double c = G[g]->center[j], e = fmax(fabs(pool.lo[j] - c), fabs(pool.lo[j] + pool.span[j] - c));
          a2[g] += (e / G[g]->ell[j]) * (e / G[g]->ell[j]);
        }
  } else {                                                          // FP32 is plenty for a launch choice
    float inv[2][12];
    for (int g = 0; g < 2; ++g)
      for (int j = 0; j < 12; ++j) inv[g][j] = j < d ? (float)(1.0 / G[g]->ell[j]) : 0.f;
    for (long long r = t0; r < m; r += stride) {
      float s0 = 0.f, s1 = 0.f;
      for (int j = 0; j < d; ++j) {
        const float a = (float)ombo_pool_coord(pool, r, j);
        const float e0 = (a - (float)G[0]->center[j]) * inv[0][j], e1 = (a - (float)G[1]->center[j]) * inv[1][j];
        s0 = fmaf(e0, e0, s0);
        s1 = fmaf(e1, e1, s1);
      }
      a2[0] = fmax(a2[0], (double)s0);
      a2[1] = fmax(a2[1], (double)s1);
    }
  }
  for (int g = 0; g < 2; ++g) {
    atomicMax(&ext[g], (unsigned long long)__double_as_longlong(a2[g]));
    atomicMax(&ext[2 + g], (unsigned long long)__double_as_longlong(b2[g]));
  }
}

static void stage1_gp(Stage1Gp &q, const GpDev &g) {
  q.xs32 = g.xs32; q.alpha32 = g.alpha32; q.b2_32 = g.b2_32;
  q.ell = g.ell; q.center = g.center;
  q.n_pad = g.n_pad;
  q.var_up = (float)(fmax(g.sigma_f2, g.var_floor) + g.sigma_n2);   // as ombo_mean8_bound
  q.matern = g.kernel == OMBO_KERNEL_MATERN52;
}

int ombo_stage1_tc_useful(ombo_ctx *ctx, const GpDev gp[2], const PoolDev &pool, long long m, void *ws, bool *useful,
                          cudaStream_t s) {
  Stage1Gp q[2];
  stage1_gp(q[0], gp[0]);
  stage1_gp(q[1], gp[1]);
  unsigned long long *ext = (unsigned long long *)ws;
  OMBO_CUDA(cudaMemsetAsync(ext, 0, 4 * sizeof(unsigned long long), s));
  const long long blocks = pool.X ? std::min((m + 255) / 256, 4LL * ctx->num_sms) : 1;
  k_stage1_extent<<<(unsigned)std::max(1LL, blocks), 256, 0, s>>>(q[0], q[1], pool, m, gp[0].d, ext);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  static_assert(4 * sizeof(double) <= 64, "the extents are read back through the context's 64-byte pinned buffer");
  OMBO_CUDA(cudaMemcpyAsync(ctx->pinned_best, ext, 4 * sizeof(double), cudaMemcpyDeviceToHost, s));
  OMBO_CUDA(cudaStreamSynchronize(s));
  double e[4];
  memcpy(e, ctx->pinned_best, sizeof(e));
  *useful = true;
  for (int g = 0; g < 2; ++g) {
    const double sa = sqrt(e[g]) + sqrt(e[2 + g]);
    double e_r;
    const double rel = s1_rel_margin(sa * sa, q[g].matern != 0, q[g].n_pad, e_r);
    *useful = *useful && rel <= S1_REL_MAX && e_r <= S1_ER_MAX;
  }
  return OMBO_OK;
}

static size_t stage1_tc_smem(int nb, int n_pf) {
  return 1024 + (size_t)nb * 128 + 2 * S1_TILE_BYTES + 4 * (size_t)nb * 4 + 2 * 4 * 4 * S1_ROWS * 4 +
         2 * (size_t)(n_pf + 2) * 4 + 16 + 48 * 8 + S1_PROD * 16 + 16 + 16 + 12 * 8 + 16;
}

bool ombo_stage1_tc_covers(const GpDev gp[2], int n_pf) {
  const int d = gp[0].d;
  const int nb = std::max(gp[0].n_pad, gp[1].n_pad);
  return d >= 1 && d <= 12 && gp[1].d == d && gp[0].n_pad % 128 == 0 && gp[1].n_pad % 128 == 0 &&
         stage1_tc_smem(nb, n_pf) <= 227 * 1024;
}

template <bool MAT0, bool MAT1>
static int launch_stage1_tc(const Stage1Params &p, size_t smem, int grid, cudaStream_t s) {
  OMBO_CUDA(cudaFuncSetAttribute(k_stage1_tc<MAT0, MAT1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_stage1_tc<MAT0, MAT1><<<grid, S1_THREADS, smem, s>>>(p);
  OMBO_CUDA(cudaGetLastError());
  return OMBO_OK;
}

int ombo_stage1_tc_bound(ombo_ctx *ctx, const GpDev gp[2], const PoolDev &pool, long long m, const double *stripes,
                         int n_pf, float c00, float c01, double *ub, ombo_best *best_dev, double *mu_out,
                         double *marg_out, int *grid_out, cudaStream_t s) {
  if (!ombo_stage1_tc_covers(gp, n_pf)) { ombo_set_error("stage1_tc: shape not covered"); return OMBO_ERR_UNSUPPORTED; }
  Stage1Params p;
  memset(&p, 0, sizeof(p));
  for (int g = 0; g < 2; ++g) stage1_gp(p.gp[g], gp[g]);
  p.pool = pool; p.m = m; p.d = gp[0].d; p.n_pf = n_pf; p.c00 = c00; p.c01 = c01;
  p.nb = std::max(gp[0].n_pad, gp[1].n_pad);
  p.stripes = stripes; p.ub = ub; p.mu_out = mu_out; p.marg_out = marg_out;
  const long long tiles = (m + S1_ROWS - 1) / S1_ROWS;
  const int grid = (int)std::max(1LL, std::min(tiles, (long long)ctx->num_sms));
  if (grid_out) *grid_out = grid;
  int rc = ombo_ws_reserve(&ctx->ws_partial, &ctx->ws_partial_bytes, (size_t)grid * sizeof(ombo_best));
  if (rc) return rc;
  p.partials = (ombo_best *)ctx->ws_partial;
  const size_t smem = stage1_tc_smem(p.nb, n_pf);
  const bool m0 = p.gp[0].matern, m1 = p.gp[1].matern;
  {
    ProfScope prof(ctx, s);
    rc = m0 ? (m1 ? launch_stage1_tc<true, true>(p, smem, grid, s) : launch_stage1_tc<true, false>(p, smem, grid, s))
            : (m1 ? launch_stage1_tc<false, true>(p, smem, grid, s) : launch_stage1_tc<false, false>(p, smem, grid, s));
  }
  if (rc) return rc;
  ctx->launches += 1;
  return ombo_argmax_merge(ctx, grid, best_dev, s);
}
