// Per-candidate acquisition arithmetic shared by K4 (acquisition.cu) and by the fast posterior kernel's fused
// epilogue (posterior_fast8.cu): the normal cdf / pdf pair and the closed-form 2-D EHVI.
// Restates util_functions.py:136-167 (EHVI) + :81-128 (EHVI_2D_aux) + :130-133 (psi_cal) of the reference tree.
#pragma once

__device__ __forceinline__ double Phi(double t) { return 0.5 * erfc(-t * 0.70710678118654752440); }
__device__ __forceinline__ double phi(double t) { return exp(-(t * t) / 2.0) / 2.50662827463100050242; }
// FP32 twins for the fast precision mode (tolerance 1e-3): erfcf keeps its relative accuracy in the tails,
// exp goes through MUFU.EX2 -- the FP64 pipe of the B200 is ~60x narrower than the FP32 one
__device__ __forceinline__ float Phi(float t) { return 0.5f * erfcf(-t * 0.70710678f); }
__device__ __forceinline__ float phi(float t) { return __expf(-0.5f * t * t) * 0.39894228f; }
__device__ __forceinline__ float sqrt_t(float x) { return sqrtf(x); }
__device__ __forceinline__ double sqrt_t(double x) { return sqrt(x); }
__device__ __forceinline__ float fmax_t(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double fmax_t(double a, double b) { return fmax(a, b); }

// h(t) = phi(t) + t Phi(t) = E[(t - z)^+] for z ~ N(0, 1) (EI / sigma, psi / sigma), FP32.  Below t = -5 the two terms
// cancel (h ~ phi / t^2), and near t = -13 phi flushes while t Phi(t) does not, so h turns negative.  There
// h = phi(t) q / (x + q), x = -t, with q = 1 / (x + 2 / (x + 3 / (x + ... 8 / x))) the Mills-ratio continued fraction
// cut at depth 8, evaluated by its convergents A / B (all terms positive, one division): q / (x + q) = B / (x A + B),
// relative error 3e-7 for x >= 5.  x is capped at 40, where phi has long flushed (A ~ x^8 stays finite); h flushes to 0
// with phi, near t = -13.2.
__device__ __forceinline__ float h_norm(float t) {
  if (!(t < -5.f)) return phi(t) + t * Phi(t);
  const float x = fminf(-t, 40.f);
  float a0 = 1.f, a1 = x, b0 = 0.f, b1 = 1.f;
#pragma unroll
  for (int k = 2; k <= 8; ++k) {
    const float a2 = fmaf(x, a1, (float)k * a0), b2 = fmaf(x, b1, (float)k * b0);
    a0 = a1; a1 = a2; b0 = b1; b1 = b2;
  }
  return phi(t) * __fdividef(b1, fmaf(x, a1, b1));
}

// Phi(t) as a double: below t = -5 in FP64, so that a product of several small probabilities (constrained EI) keeps
// its value below FLT_MIN instead of flushing to 0
__device__ __forceinline__ double Phi_wide(double t) { return Phi(t); }
__device__ __forceinline__ double Phi_wide(float t) { return t < -5.f ? Phi((double)t) : (double)Phi(t); }

// y1 / y2: the P + 2 stripe bounds per objective (host_prep.ehvi_stripes: front sorted by f1, reference point and
// ideal sentinel at the ends).  exact = 0: the reference's arithmetic ('sigma' = model 0's variance times the
// flattened sample covariance, util_functions.py:163,167,:115; P stripes); exact = 1: each model's own standard
// deviation and the (P+1)-th stripe the reference drops (y1[P+1] = -inf taken as a limit).
template <typename T>
__device__ __forceinline__ T ehvi2d_value(T m0, T m1, T v0, T v1, const T *__restrict__ y1, const T *__restrict__ y2,
                                          int P, bool exact, T c00, T c01) {
  const T s0 = exact ? sqrt_t(v0) : v0 * c00;
  const T s1 = exact ? sqrt_t(v1) : v0 * c01;
  T sum1 = 0, sum2 = 0;
  T tp = (y1[0] - m0) / s0;
  T cdf_p = Phi(tp), pdf_p = phi(tp);
  for (int i = 1; i <= P; ++i) {
    T t = (y1[i] - m0) / s0;
    T cdf_t = Phi(t), pdf_t = phi(t);
    T t2 = (y2[i] - m1) / s1;
    T psi2 = s1 * phi(t2) + (y2[i] - m1) * Phi(t2);
    sum1 = sum1 + (y1[i - 1] - y1[i]) * cdf_t * psi2;
    T psi_a = s0 * pdf_p + (y1[i - 1] - m0) * cdf_p;
    T psi_b = s0 * pdf_t + (y1[i - 1] - m0) * cdf_t;
    sum2 = sum2 + (psi_a - psi_b) * psi2;
    cdf_p = cdf_t; pdf_p = pdf_t;
  }
  if (exact) {
    T t2 = (y2[P + 1] - m1) / s1;
    T psi2 = s1 * phi(t2) + (y2[P + 1] - m1) * Phi(t2);
    T psi_a = s0 * pdf_p + (y1[P] - m0) * cdf_p;
    sum2 = sum2 + psi_a * psi2;
  }
  return sum1 + sum2;
}

// FP32 (fast precision mode, K4 and the fused f8c epilogue): the same value rearranged so that no step cancels.  With
// t_i = (y1[i] - m0) / s0, psi(y1[i-1], y1[i-1]) = s0 h(t_{i-1}) and psi(y1[i-1], y1[i]) = s0 h(t_i) + (y1[i-1] - y1[i])
// Phi(t_i), so sum1 + sum2 = s0 sum_i (h(t_{i-1}) - h(t_i)) psi2_i with psi2_i = s1 h(t2_i).  h is taken tail-safe
// (h_norm) and split as h(t) = max(t, 0) + h(-|t|), so the difference is (max(t_{i-1}, 0) - max(t_i, 0)) +
// h(-|t_{i-1}|) - h(-|t_i|); where both t are >= 0 the first part is taken as (y1[i-1] - y1[i]) / s0, so a stripe far
// above the mean is not a difference of two numbers ~ t.  Nothing assumes y1 to decrease: a front point beyond r or a
// dominated / duplicate point gives the same value as the formula.  Values below FLT_MIN (every candidate ~9 sigma
// behind the front in both objectives) flush to 0.
template <>
__device__ __forceinline__ float ehvi2d_value<float>(float m0, float m1, float v0, float v1,
                                                     const float *__restrict__ y1, const float *__restrict__ y2, int P,
                                                     bool exact, float c00, float c01) {
  const float s0 = exact ? sqrtf(v0) : v0 * c00;
  const float s1 = exact ? sqrtf(v1) : v0 * c01;
  const float r0 = 1.f / s0;
  float tp = (y1[0] - m0) * r0;
  float gp = h_norm(-fabsf(tp));                    // h(-|t|): h(t) itself below the mean, h(t) - t above it
  float sum = 0.f;
  for (int i = 1; i <= P; ++i) {
    const float t = (y1[i] - m0) * r0;
    const float g = h_norm(-fabsf(t));
    const float lead = (t >= 0.f && tp >= 0.f) ? (y1[i - 1] - y1[i]) * r0 : fmaxf(tp, 0.f) - fmaxf(t, 0.f);
    const float psi2 = s1 * h_norm((y2[i] - m1) / s1);
    sum = fmaf(lead + (gp - g), psi2, sum);
    tp = t; gp = g;
  }
  if (exact) sum = fmaf(fmaxf(tp, 0.f) + gp, s1 * h_norm((y2[P + 1] - m1) / s1), sum);
  return s0 * sum;
}

// arg-max pair: ties resolve to the lowest global index (np.argmax)
struct BestPair { double v; long long i; };
__device__ __forceinline__ bool better(double v, long long i, double bv, long long bi) {
  return (v > bv) || (v == bv && i < bi);
}
__device__ __forceinline__ BestPair warp_best(BestPair b) {
  for (int o = 16; o; o >>= 1) {
    double ov = __shfl_xor_sync(0xffffffffu, b.v, o);
    long long oi = __shfl_xor_sync(0xffffffffu, b.i, o);
    if (better(ov, oi, b.v, b.i)) { b.v = ov; b.i = oi; }
  }
  return b;
}
