// The K1 generator arithmetic of the f8c kernel (posterior_fast8.cu), shared with the mean-only bound kernel of the
// pruned arg-max (posterior_mean8.cu).  Both kernels call exactly these functions, in the same order per (row, column
// group), so that the mean of a candidate is the same FP32 number in both -- the pruned arg-max relies on that.
//   candidate prep  x_j = -2 (a_j - c_j) / ell_j in FP32 (FP64 subtraction and scaling), a2 = |x|^2 / 4
//   dist2           r^2 of ROWS rows to the eight training points of one column group: |b|^2 + a2 + sum_j x_j b_j
//   kval            k'(r) of one row (Matern-5/2 or RBF, MUFU approximations)
//   mean_add        the row's share of the mean: sum of k' (sigma_f2 alpha) over the eight columns, into one FP32 sum
// A training slice holds DP coordinate rows, sigma_f2 alpha and |b|^2 of one 64-column K-block, 64 floats each.
#pragma once
#include "candidates.cuh"

// a candidate coordinate a (ombo_pool_coord), centred and length-scaled as the generators take it
__device__ __forceinline__ float gen8_coord(double a, double center, double inv_ell) {
  return -2.0f * (float)((a - center) * inv_ell);
}

// one candidate row into registers (coordinate j at src[j * stride]); returns a2
template <int DP>
__device__ __forceinline__ float gen8_load_row(const float *src, int stride, float (&xr)[DP]) {
  float acc = 0.f;
#pragma unroll
  for (int j = 0; j < DP; ++j) { xr[j] = src[j * stride]; acc = fmaf(xr[j], xr[j], acc); }
  return 0.25f * acc;
}

// xs: the slice offset by this lane's column group (8 g)
template <int DP, int ROWS>
__device__ __forceinline__ void gen8_dist2(const float *xs, const float (&x)[ROWS][DP], const float (&a2)[ROWS],
                                           float2 (&r2)[ROWS][4]) {
  {
    const float4 n0 = *(const float4 *)(xs + (DP + 1) * 64);      // |b_i|^2
    const float4 n1 = *(const float4 *)(xs + (DP + 1) * 64 + 4);
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) {
      const float2 aa = make_float2(a2[rr], a2[rr]);
      r2[rr][0] = __fadd2_rn(aa, make_float2(n0.x, n0.y));
      r2[rr][1] = __fadd2_rn(aa, make_float2(n0.z, n0.w));
      r2[rr][2] = __fadd2_rn(aa, make_float2(n1.x, n1.y));
      r2[rr][3] = __fadd2_rn(aa, make_float2(n1.z, n1.w));
    }
  }
#pragma unroll
  for (int j = 0; j < DP; ++j) {
    const float4 t0 = *(const float4 *)(xs + j * 64);
    const float4 t1 = *(const float4 *)(xs + j * 64 + 4);
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) {
      const float2 xx = make_float2(x[rr][j], x[rr][j]);            // -2 a_j
      r2[rr][0] = __ffma2_rn(xx, make_float2(t0.x, t0.y), r2[rr][0]);
      r2[rr][1] = __ffma2_rn(xx, make_float2(t0.z, t0.w), r2[rr][1]);
      r2[rr][2] = __ffma2_rn(xx, make_float2(t1.x, t1.y), r2[rr][2]);
      r2[rr][3] = __ffma2_rn(xx, make_float2(t1.z, t1.w), r2[rr][3]);
    }
  }
}

template <bool MATERN>
__device__ __forceinline__ void gen8_kval(const float2 (&r2r)[4], float2 (&kv)[4]) {
  if (MATERN) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float2 rad, ex;
      asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad.x) : "f"(fabsf(r2r[e].x)));
      asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad.y) : "f"(fabsf(r2r[e].y)));
      const float2 arg = __fmul2_rn(rad, make_float2(-3.2259955597f, -3.2259955597f));   // -sqrt5 log2(e)
      asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex.x) : "f"(arg.x));
      asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex.y) : "f"(arg.y));
      const float2 poly = __ffma2_rn(rad, make_float2(2.2360679775f, 2.2360679775f),
                                     __ffma2_rn(r2r[e], make_float2(1.6666666667f, 1.6666666667f),
                                                make_float2(1.0f, 1.0f)));
      kv[e] = __fmul2_rn(poly, ex);
    }
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 arg = __fmul2_rn(r2r[e], make_float2(-0.7213475204f, -0.7213475204f));  // -0.5 log2(e)
      asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(kv[e].x) : "f"(arg.x));
      asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(kv[e].y) : "f"(arg.y));
    }
  }
}

__device__ __forceinline__ void gen8_mean_add(const float2 (&kv)[4], const float4 al0, const float4 al1, float &acc) {
  float2 m2 = __fmul2_rn(kv[0], make_float2(al0.x, al0.y));
  m2 = __ffma2_rn(kv[1], make_float2(al0.z, al0.w), m2);
  m2 = __ffma2_rn(kv[2], make_float2(al1.x, al1.y), m2);
  m2 = __ffma2_rn(kv[3], make_float2(al1.z, al1.w), m2);
  acc += m2.x + m2.y;
}

// the mean of a row from its four column-pair partials (each the lane pair's sum, acc + shfl_xor(acc, 1))
__device__ __forceinline__ float gen8_mean_sum(float p0, float p1, float p2, float p3) { return (p0 + p1) + (p2 + p3); }
