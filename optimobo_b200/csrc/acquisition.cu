// K4 + K5 -- per-candidate acquisition value from the GP posteriors, and the arg-max.
// One thread per candidate, FP64 throughout (the reference is float64 numpy/scipy); the sorted
// Pareto-front stripes / cells / cached samples are staged in shared memory once per block.
//
// Formulas restate (file:line into the reference tree, optimobo/):
//   EHVI2D            util_functions.py:136-167 (EHVI) + :81-128 (EHVI_2D_aux) + :130-133 (psi_cal)
//   EHVI3D            util_functions.py:170-214
//   EXPECTED_DECOMP   util_functions.py:285-327 with the 12 scalarisations of scalarisations.py
//   EI                optimisers.py:325-344, parego.py:126-145, keep.py:118-137, cparego.py:450-469
//   CONSTRAINED_EI    cparego.py:471-496
//   PARETO_EI         keep.py:142-150
//   HV_POI            emo.py:176-228
//   EHVI_BOX          not in the reference: the exact k-objective EHVI over a box decomposition (k_acquire_box)
//   EHVI_BOX_FEAS     not in the reference: EHVI_BOX times the probability of feasibility of CONSTRAINED_EI
//   HV_POI_BOX        HV_POI for 2 to 4 objectives: the same region, tiled by the boxes of EHVI_BOX (k_acquire_box)
// Arg-max replaces the inner optimiser call sites (differential_evolution at optimisers.py:87,
// :118,:366; cparego.py:94,:544; emo.py:240; EA loops parego.py:242-270, keep.py:260-292):
// warp shuffle -> block (smem) -> per-block partial -> one final block; ties resolve to the
// lowest global index (np.argmax), NaN is treated as -inf.
#include "common.cuh"
#include "acq_math.cuh"

#define ACQ_THREADS 256


// ---- scalarisations (scalarisations.py) --------------------------------------------------
__device__ double scalarise(const ombo_acq &a, const double *F) {
  const int k = a.n_obj;
  double Fp[OMBO_MAX_OBJ];
  for (int i = 0; i < k; ++i) Fp[i] = (F[i] - a.ideal[i]) / (a.maxp[i] - a.ideal[i]);
  const double *w = a.weights;
  switch (a.scalarisation) {
    case OMBO_SC_WEIGHTED_SUM: {            // :43-50
      double s = 0.0;
      for (int i = 0; i < k; ++i) s += Fp[i] * w[i];
      return s;
    }
    case OMBO_SC_TCHEBICHEFF: {             // :66-72
      double mx = w[0] * Fp[0];
      for (int i = 1; i < k; ++i) mx = fmax(mx, w[i] * Fp[i]);
      return mx;
    }
    case OMBO_SC_AUG_TCHEBICHEFF: {         // :92-109
      double mx = fabs(Fp[0]) * w[0], sum = fabs(Fp[0]);
      for (int i = 1; i < k; ++i) { mx = fmax(mx, fabs(Fp[i]) * w[i]); sum += fabs(Fp[i]); }
      return mx + a.sc_params[0] * sum;
    }
    case OMBO_SC_MOD_TCHEBICHEFF: {         // :130-149
      double sum = 0.0;
      for (int i = 0; i < k; ++i) sum += fabs(Fp[i]);
      double right = a.sc_params[0] * sum;
      double mx = (fabs(Fp[0]) + right) * w[0];
      for (int i = 1; i < k; ++i) mx = fmax(mx, (fabs(Fp[i]) + right) * w[i]);
      return mx;
    }
    case OMBO_SC_EXP_WEIGHTED: {            // :165-173
      double s = 0.0, p = a.sc_params[0];
      for (int i = 0; i < k; ++i) s += exp(p * w[i] - 1.0) * exp(p * Fp[i]);
      return s;
    }
    case OMBO_SC_WEIGHTED_NORM: {           // :190-197
      double s = 0.0, p = a.sc_params[0];
      for (int i = 0; i < k; ++i) s += pow(fabs(Fp[i]), p) * w[i];
      return pow(s, 1.0 / p);
    }
    case OMBO_SC_WEIGHTED_POWER: {          // :212-219
      double s = 0.0, p = a.sc_params[0];
      for (int i = 0; i < k; ++i) s += pow(Fp[i], p) * w[i];
      return s;
    }
    case OMBO_SC_WEIGHTED_PRODUCT: {        // :230-238
      double s = 1.0;
      for (int i = 0; i < k; ++i) s *= pow(Fp[i] + 100000.0, w[i]);
      return s;
    }
    case OMBO_SC_PBI:
    case OMBO_SC_IPBI:
    case OMBO_SC_QPBI: {                    // :257-273, :291-310, :325-351
      double nw = 0.0;
      for (int i = 0; i < k; ++i) nw += w[i] * w[i];
      nw = sqrt(nw);
      double d1 = 0.0;
      for (int i = 0; i < k; ++i) d1 += Fp[i] * (w[i] / nw);
      double d2 = 0.0;
      for (int i = 0; i < k; ++i) { double e = Fp[i] - d1 * (w[i] / nw); d2 += e * e; }
      d2 = sqrt(d2);
      const double theta = a.sc_params[0];
      if (a.scalarisation == OMBO_SC_PBI) return d1 + theta * d2;
      if (a.scalarisation == OMBO_SC_IPBI) return theta * d2 - d1;
      double span = 0.0;
      for (int i = 0; i < k; ++i) span += a.maxp[i] - a.ideal[i];
      double d_star = a.sc_params[1] * ((1.0 / a.sc_params[2]) * (1.0 / (double)k) * span);
      return d1 + theta * d2 * (d2 / d_star);
    }
    case OMBO_SC_APD: {                     // :375-397
      double nf = 0.0;
      bool allz = true, wz = true;
      for (int i = 0; i < k; ++i) { nf += Fp[i] * Fp[i]; allz = allz && (Fp[i] == 0.0); wz = wz && (w[i] == 0.0); }
      nf = sqrt(nf);                        // norm taken before the 1e-5 patch (:384)
      double n1 = 0.0, n2 = 0.0, dot = 0.0;
      double f[OMBO_MAX_OBJ], ww[OMBO_MAX_OBJ];
      for (int i = 0; i < k; ++i) { f[i] = allz ? 1e-5 : Fp[i]; ww[i] = wz ? 1e-5 : w[i]; n1 += f[i] * f[i]; n2 += ww[i] * ww[i]; }
      n1 = sqrt(n1); n2 = sqrt(n2);
      for (int i = 0; i < k; ++i) dot += (f[i] / n1) * (ww[i] / n2);
      double th = acos(fmin(1.0, fmax(-1.0, dot)));
      return (1.0 + (double)k * (a.sc_params[0] / a.sc_params[1]) * (th / a.sc_params[2])) * nf;
    }
  }
  return nan("");
}

// ---- EI ----------------------------------------------------------------------------------
// T = float: best - mu and var + eps are formed in FP64 before the cast (a pool far from the origin keeps the digits of
// its spread), and below g = -5, where g Phi(g) + phi(g) cancels and then flushes, the lane switches to FP64: the
// result is a double, so EI down to ~1e-300 (g ~ -37) survives.  Natural pools rarely have such lanes.
template <typename T>
__device__ __forceinline__ double ei_value(double mu, double var, double best, double eps) {
  T s = sqrt_t((T)(var + eps));
  T g = (T)(best - mu) / (s + (T)1e-10);
  if (sizeof(T) == sizeof(double) || !(g < (T)-5)) return s * (g * Phi(g) + phi(g));
  const double sd = sqrt(var + eps), gd = (best - mu) / (sd + 1e-10);
  return fmax(sd * (gd * Phi(gd) + phi(gd)), 0.0);       // below g ~ -37 the FP64 terms cancel to +-subnormals
}

extern __shared__ __align__(16) double acq_smem[];

// T = double: the reference's arithmetic (FP64 precision mode, all goldens).  T = float: the fast precision mode
// (tolerance 1e-3) -- same formulas on the FP32 pipe with erfcf / MUFU exp; the expected decomposition always runs
// in double (ExponentialWeightedCriterion overflows FP32, WeightedProduct's 1e5 offset eats its digits).
template <typename T>
__global__ void __launch_bounds__(ACQ_THREADS)
k_acquire(ombo_acq a, int n_gp, const double *__restrict__ mu, const double *__restrict__ var,
          long long m, long long ld, long long index_base, double *__restrict__ out_acq,
          ombo_best *__restrict__ partials) {
  // stage the per-iteration constants
  T *cst = reinterpret_cast<T *>(acq_smem);
  int n_stage = 0;
  const double *src = nullptr;
  if (a.kind == OMBO_ACQ_EHVI2D) { n_stage = 2 * (a.n_pf + 2); src = a.stripes; }
  else if (a.kind == OMBO_ACQ_HV_POI) { n_stage = a.n_cells * 2 * a.n_obj; src = a.cells; }
  else if (a.kind == OMBO_ACQ_EHVI3D || a.kind == OMBO_ACQ_EXPECTED_DECOMP) { n_stage = a.n_samples * a.n_obj; src = a.cache; }
  for (int e = threadIdx.x; e < n_stage; e += ACQ_THREADS) cst[e] = (T)src[e];
  __syncthreads();

  const long long c = (long long)blockIdx.x * ACQ_THREADS + threadIdx.x;
  double val = -INFINITY;
  if (c < m) {
    T mus[OMBO_MAX_GP], vars[OMBO_MAX_GP];
    for (int g = 0; g < n_gp; ++g) { mus[g] = (T)mu[g * ld + c]; vars[g] = (T)var[g * ld + c]; }
    double r = nan("");
    switch (a.kind) {
      case OMBO_ACQ_EHVI2D: {
        const int P = a.n_pf;
        r = ehvi2d_value<T>(mus[0], mus[1], vars[0], vars[1], cst, cst + (P + 2), P, a.semantics == OMBO_SEM_EXACT,
                            (T)a.cache_c00, (T)a.cache_c01);
      } break;
      case OMBO_ACQ_EHVI3D:
      case OMBO_ACQ_EXPECTED_DECOMP: {
        const int k = a.n_obj, S = a.n_samples;
        const bool exact = (a.semantics == OMBO_SEM_EXACT);
        T sd[OMBO_MAX_OBJ];
        for (int i = 0; i < k; ++i) sd[i] = sqrt_t(exact ? vars[i] : vars[0]);   // util_functions.py:233
        T total = 0;
        for (int j = 0; j < S; ++j) {
          T Y[OMBO_MAX_OBJ];
          for (int i = 0; i < k; ++i) Y[i] = cst[j * k + i] * sd[i] + mus[i];
          if (a.kind == OMBO_ACQ_EHVI3D) {
            bool inside = true;
            T hv = 1;
            for (int i = 0; i < k; ++i) { T df = (T)a.ref[i] - Y[i]; inside = inside && (df >= (T)0); hv = (i == 0) ? df : hv * df; }
            hv -= (T)a.best;    // Sminus = HV(PF), hoisted (util_functions.py:198-199)
            if (inside && hv > (T)0) total += hv;
          } else {
            double Yd[OMBO_MAX_OBJ];
            for (int i = 0; i < k; ++i) Yd[i] = (double)Y[i];
            double g = scalarise(a, Yd);
            total += (T)fmax(0.0, a.best - g);
            if (isnan(g)) total = (T)nan("");
          }
        }
        r = total / (T)S;
      } break;
      // the EI family reads its inputs as doubles (ei_value)
      case OMBO_ACQ_EI:
        r = ei_value<T>(mu[c], var[c], a.best, a.var_eps[0]);
        break;
      case OMBO_ACQ_CONSTRAINED_EI: {
        r = ei_value<T>(mu[c], var[c], a.best, a.var_eps[0]);
        double pof = 1;           // a mostly infeasible pool is a product of small probabilities: accumulated in FP64
        for (int g = 1; g < n_gp; ++g) pof *= Phi_wide(((T)0 - mus[g]) / sqrt_t(vars[g] + (T)a.var_eps[g]));
        r = r * pof;
      } break;
      case OMBO_ACQ_PARETO_EI:
        r = mu[c] * ei_value<T>(mu[ld + c], var[ld + c], a.best, a.var_eps[1]);
        break;
      case OMBO_ACQ_HV_POI: {
        const int k = 2;     // emo.py:21 "Only works for 2D so far"
        T sd[2];
        for (int i = 0; i < k; ++i) sd[i] = sqrt_t(vars[i] + (T)a.var_eps[i]);
        T poi = 0, imp = 0;
        for (int cix = 0; cix < a.n_cells; ++cix) {
          const T *U = cst + (size_t)cix * 2 * a.n_obj, *Lo = U + a.n_obj;
          T p = 1, vol = 1;
          bool valid = true;
          for (int i = 0; i < k; ++i) {
            const T za = (U[i] - mus[i]) / sd[i], zb = (Lo[i] - mus[i]) / sd[i];
            // FP32: a cell above the mean (za > zb > 0) takes the difference of the two upper tails, which keeps its
            // digits where Phi(za) - Phi(zb) is a difference of two numbers near 1
            T pi = (sizeof(T) == sizeof(float) && zb > (T)0) ? Phi(-zb) - Phi(-za) : Phi(za) - Phi(zb);
            p = (i == 0) ? pi : p * pi;
            valid = valid && (U[i] > mus[i]);
            T e = U[i] - fmax_t(Lo[i], mus[i]);
            vol = (i == 0) ? e : vol * e;
          }
          poi += p;
          if (valid) imp += vol;
        }
        r = poi * imp;
      } break;
      default:
        r = 0;
    }
    if (out_acq) out_acq[c] = (double)r;
    val = isnan(r) ? -INFINITY : (double)r;
  }
  // ---- K5: block arg-max ----
  BestPair b;
  b.v = val;
  b.i = (c < m) ? index_base + c : 0x7fffffffffffffffLL;
  b = warp_best(b);
  __shared__ double sv[ACQ_THREADS / 32];
  __shared__ long long si[ACQ_THREADS / 32];
  if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = b.v; si[threadIdx.x >> 5] = b.i; }
  __syncthreads();
  if (threadIdx.x < 32) {
    BestPair q;
    q.v = (threadIdx.x < ACQ_THREADS / 32) ? sv[threadIdx.x] : -INFINITY;
    q.i = (threadIdx.x < ACQ_THREADS / 32) ? si[threadIdx.x] : 0x7fffffffffffffffLL;
    q = warp_best(q);
    if (threadIdx.x == 0) { partials[blockIdx.x].value = q.v; partials[blockIdx.x].index = q.i; }
  }
}

// merges the per-block partials with the running best (chunks / previous passes)
__global__ void __launch_bounds__(1024) k_argmax_final(const ombo_best *__restrict__ partials, int n_partials,
                                                       ombo_best *__restrict__ best) {
  BestPair b;
  b.v = -INFINITY; b.i = 0x7fffffffffffffffLL;
  for (int e = threadIdx.x; e < n_partials; e += 1024) {
    double v = partials[e].value; long long i = partials[e].index;
    if (better(v, i, b.v, b.i)) { b.v = v; b.i = i; }
  }
  b = warp_best(b);
  __shared__ double sv[32];
  __shared__ long long si[32];
  if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = b.v; si[threadIdx.x >> 5] = b.i; }
  __syncthreads();
  if (threadIdx.x < 32) {
    BestPair q; q.v = sv[threadIdx.x]; q.i = si[threadIdx.x];
    q = warp_best(q);
    if (threadIdx.x == 0) {
      double cv = best->value; long long ci = best->index;
      if (ci < 0 || better(q.v, q.i, cv, ci)) { best->value = q.v; best->index = q.i; }
    }
  }
}

// the 12 scalarisation functions on explicit objective vectors (device twin of Scalarisation.__call__,
// scalarisations.py:20-27): out[r] = g(F[r, :], w)
__global__ void k_scalarise(ombo_acq a, const double *__restrict__ F, long long m, double *__restrict__ out) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= m) return;
  double f[OMBO_MAX_OBJ];
  for (int i = 0; i < a.n_obj; ++i) f[i] = F[r * a.n_obj + i];
  out[r] = scalarise(a, f);
}

int ombo_scalarise_impl(ombo_ctx *ctx, const ombo_acq *acq, const double *F, long long m, double *out, cudaStream_t s) {
  if (m <= 0) return OMBO_OK;
  k_scalarise<<<(unsigned)((m + 127) / 128), 128, 0, s>>>(*acq, F, m, out);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  return OMBO_OK;
}

__global__ void k_best_init(ombo_best *best) { best->value = -INFINITY; best->index = -1; }

__global__ void k_pack_key(const ombo_best *__restrict__ best, long long *__restrict__ key) {
  float f = (float)best->value;
  unsigned bits = __float_as_uint(f);
  unsigned ord = (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u);
  long long idx = best->index;
  unsigned low = (idx < 0 || idx > 0xFFFFFFFFll) ? 0u : (0xFFFFFFFFu - (unsigned)idx);
  long long hi = (long long)ord - 2147483648ll;            // signed, order-preserving
  *key = (hi << 32) | (long long)low;
}

int ombo_pack_key_impl(ombo_ctx *ctx, const ombo_best *best_dev, long long *key_dev, cudaStream_t s) {
  k_pack_key<<<1, 1, 0, s>>>(best_dev, key_dev);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  return OMBO_OK;
}

int ombo_best_init(ombo_ctx *ctx, ombo_best *best_dev, cudaStream_t s) {
  k_best_init<<<1, 1, 0, s>>>(best_dev);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  return OMBO_OK;
}

int ombo_argmax_merge(ombo_ctx *ctx, int n_partials, ombo_best *best_dev, cudaStream_t s) {
  k_argmax_final<<<1, 1024, 0, s>>>((const ombo_best *)ctx->ws_partial, n_partials, best_dev);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  return OMBO_OK;
}

// ---- K4 for OMBO_ACQ_EHVI_BOX: exact EHVI over the box decomposition -------------------------------
// A CTA of 256 threads scores a tile of `tile` candidates (32, 16 or 8, chosen from B on the host):
//   phase 1: V[cand][i][b] for every breakpoint t_b of every objective, spread over all threads (k*B Phi/phi pairs
//            per candidate);
//   phase 2: the boxes are staged BOX_CHUNK at a time as packed 16-bit indices; the G = 256 / tile slots of a
//            candidate stride over them (the lanes of a warp: one box, different candidates), each box costing k table
//            differences and multiplies; the slots are summed in a fixed order.
// V keeps H(t) = E[(t - y)^+] below the mean and (t - r) + G(t), G(t) = E[(y - t)^+] = H(t) - (t - mu), at or above
// it, so a box whose breakpoints both lie above the mean takes H(u) - H(l) = (u - l) + G(u) - G(l) without
// subtracting two numbers ~ t - mu (the FP32 cancellation); a box that straddles the mean adds back r - mu.
#define BOX_CHUNK 512

// (n_boxes, 2, k) f64 breakpoint indices -> uint4 {u0 | u1 << 16, u2 | u3 << 16, l0 | l1 << 16, l2 | l3 << 16}; an
// index outside [0, B) (or NaN) is clamped, so a malformed table cannot read past the V table
__global__ void k_pack_boxes(const double *__restrict__ cells, int n_boxes, int k, int B, uint4 *__restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_boxes) return;
  unsigned h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int s = 0; s < 2; ++s)
    for (int i = 0; i < k; ++i) {
      const double v = cells[((size_t)c * 2 + s) * k + i];
      h[s * 4 + i] = v >= 0.0 ? (v < (double)(B - 1) ? (unsigned)v : (unsigned)(B - 1)) : 0u;
    }
  out[c] = make_uint4(h[0] | h[1] << 16, h[2] | h[3] << 16, h[4] | h[5] << 16, h[6] | h[7] << 16);
}

// s h(-az) = s phi(az) - |w| Phi(-az), az = |w| / s: H(t) below the mean, G(t) above it.  FP32 takes the tail-safe
// h_norm (far from the mean the two terms cancel, and turn negative once phi flushes)
__device__ __forceinline__ double shortfall_tail(double s, double az, double w) { return s * phi(az) - fabs(w) * Phi(-az); }
__device__ __forceinline__ float shortfall_tail(float s, float az, float) { return s * h_norm(-az); }

// odd candidate stride of V (in elements): the groups of one warp read the same box from different banks
__host__ __device__ inline int box_cand_stride(int k, int B) { return (k * B) | 1; }

// feas: OMBO_ACQ_EHVI_BOX_FEAS adds the (tile,) f64 feasibility products
template <typename T>
__host__ __device__ inline size_t box_smem_bytes(int k, int B, int tile, bool feas = false) {
  return (size_t)BOX_CHUNK * 16 + (size_t)k * B * sizeof(T) + (size_t)tile * k * (3 * sizeof(T) + 4) +
         (size_t)tile * box_cand_stride(k, B) * sizeof(T) + (feas ? (size_t)tile * 8 : 0);
}

// MODE selects what the box sum adds up:
//   BOX_EHVI  (OMBO_ACQ_EHVI_BOX): the EHVI above.
//   BOX_FEAS  (OMBO_ACQ_EHVI_BOX_FEAS): GPs K..n_gp-1 are constraint models, and the value is the box sum times the
//             probability of feasibility prod_j Phi(-mu_j / sqrt(var_j + var_eps[j])), formed in FP64 exactly as the
//             constrained EI forms it (k_acquire), once per candidate in the prologue.
//   BOX_HVPOI (OMBO_ACQ_HV_POI_BOX): the table's index 0 is the ideal point, sigma = sqrt(var + var_eps), and the
//             value is PoI * Imp with PoI = sum_c prod_i P(l_ci < y_i <= u_ci) and Imp = sum_c prod_i
//             (max(u_ci - mu_i, 0) - max(l_ci - mu_i, 0)).  V keeps Phi(z) below the mean and Phi(z) - 1 = -Phi(-z) at
//             or above it, so a box above the mean takes Phi(-z_l) - Phi(-z_u) (two upper tails, not two numbers
//             near 1) and a box that straddles the mean adds back 1.  The extents come from the t - r row and r - mu;
//             a box above the mean takes (u - r) - (l - r), not a difference of two numbers ~ t - mu.
enum { BOX_EHVI = 0, BOX_FEAS = 1, BOX_HVPOI = 2 };

template <typename T, int K, int MODE>
__global__ void __launch_bounds__(ACQ_THREADS)
k_acquire_box(ombo_acq a, int tile, const double *__restrict__ mu, const double *__restrict__ var, long long m,
              long long ld, long long index_base, const uint4 *__restrict__ boxes, double *__restrict__ out_acq,
              ombo_best *__restrict__ partials, int n_gp) {
  constexpr bool FEAS = MODE == BOX_FEAS, HVPOI = MODE == BOX_HVPOI;
  const int B = a.n_pf, n_boxes = a.n_cells, G = ACQ_THREADS / tile, cs = box_cand_stride(K, B);
  uint4 *bx = reinterpret_cast<uint4 *>(acq_smem);                  // BOX_CHUNK staged boxes
  double *pof = reinterpret_cast<double *>(bx + BOX_CHUNK);         // FEAS: (tile,) feasibility products
  T *V = reinterpret_cast<T *>(pof + (FEAS ? tile : 0));            // (tile, cs)
  T *tr = V + tile * cs;                                            // (K, B) breakpoints t - r
  T *sd = tr + K * B;                                               // (tile, K) sigma
  T *rsd = sd + tile * K;                                           // (tile, K) 1 / sigma
  T *shift = rsd + tile * K;                                        // (tile, K) r - mu
  int *split = reinterpret_cast<int *>(shift + tile * K);           // (tile, K) first b with t_b - mu >= 0
  const long long c0 = (long long)blockIdx.x * tile;

  // the only FP64 arithmetic: t - r once per CTA and r - mu once per candidate and objective, so that t - mu =
  // (t - r) + (r - mu) keeps its digits in FP32 when the front sits far from the origin (the FP64 pipe is narrow)
  for (int e = threadIdx.x; e < K * B; e += ACQ_THREADS) tr[e] = (T)(a.stripes[e] - a.stripes[(e / B) * B + B - 1]);
  for (int e = threadIdx.x; e < tile * K; e += ACQ_THREADS) {
    const int j = e / K, i = e - j * K;
    const long long c = c0 + j;
    const double mv = c < m ? mu[i * ld + c] : 0.0, vv = c < m ? var[i * ld + c] : 1.0;
    sd[e] = HVPOI ? sqrt_t((T)(vv + a.var_eps[i])) : sqrt_t((T)vv);
    rsd[e] = (T)1 / sd[e];
    shift[e] = (T)(a.stripes[i * B + B - 1] - mv);
    split[e] = B;                                                   // mu above every breakpoint
  }
  if (FEAS)
    for (int j = threadIdx.x; j < tile; j += ACQ_THREADS) {
      const long long c = c0 + j;
      double p = 1;           // a mostly infeasible pool is a product of small probabilities: accumulated in FP64
      if (c < m)
        for (int g = K; g < n_gp; ++g)
          p *= Phi_wide(((T)0 - (T)mu[g * ld + c]) / sqrt_t((T)var[g * ld + c] + (T)a.var_eps[g]));
      pof[j] = p;
    }
  __syncthreads();
  // phase 1: the V table
  for (int e = threadIdx.x; e < tile * K * B; e += ACQ_THREADS) {
    const int j = e / (K * B), ib = e - j * (K * B), i = ib / B, b = ib - i * B, jk = j * K + i;
    T v = 0;                                                        // H(-inf) = 0
    if constexpr (HVPOI) {                                          // index 0 is the ideal point: evaluated too
      const T c = shift[jk], w = tr[ib] + c;                        // t - mu
      const T z = w * rsd[jk];
      v = w >= (T)0 ? -Phi(-z) : Phi(z);
      if (w >= (T)0 && (b == 0 || tr[ib - 1] + c < (T)0)) split[jk] = b;
    } else if (b > 0) {
      const T c = shift[jk], s = sd[jk];
      const T w = tr[ib] + c;                                       // t - mu
      const T az = fabs(w * rsd[jk]);
      const T g = shortfall_tail(s, az, w);                         // H(t) below the mean, G(t) above
      v = w >= (T)0 ? tr[ib] + g : g;
      if (tr[ib - 1] + c < (T)0 && w >= (T)0) split[jk] = b;        // one writer: t - mu is nondecreasing in b
    }
    V[j * cs + ib] = v;
  }
  __syncthreads();
  // phase 2: the box sum.  Thread = (slot, candidate j): the lanes of a warp share a slot (tile 32; two slots at tile
  // 16, four at 8), so they read one broadcast box and gather V of different candidates through the odd stride
  const int j = threadIdx.x % tile, slot = threadIdx.x / tile;
  const long long c = c0 + j;
  T shj[K];
  int spj[K];
#pragma unroll
  for (int i = 0; i < K; ++i) { shj[i] = shift[j * K + i]; spj[i] = split[j * K + i]; }
  const T *Vj = V + j * cs;
  T acc = 0, vol = 0;                                               // HVPOI: the PoI and the Imp sums
  for (int base = 0; base < n_boxes; base += BOX_CHUNK) {
    const int n = min(BOX_CHUNK, n_boxes - base);
    for (int e = threadIdx.x; e < n; e += ACQ_THREADS) bx[e] = boxes[base + e];
    __syncthreads();
    if (c < m) {
      for (int q = slot; q < n; q += G) {
        const uint4 p = bx[q];
        const unsigned uu[4] = {p.x & 0xffffu, p.x >> 16, p.y & 0xffffu, p.y >> 16};
        const unsigned ll[4] = {p.z & 0xffffu, p.z >> 16, p.w & 0xffffu, p.w >> 16};
        T prod = 1, ext = 1;
#pragma unroll
        for (int i = 0; i < K; ++i) {
          const int u = (int)uu[i], l = (int)ll[i];
          T d = Vj[i * B + u] - Vj[i * B + l];
          if (l < spj[i] && u >= spj[i]) d += HVPOI ? (T)1 : shj[i];
          prod = i == 0 ? d : prod * d;
          if constexpr (HVPOI) {
            const T x = l >= spj[i] ? tr[i * B + u] - tr[i * B + l] : (u >= spj[i] ? tr[i * B + u] + shj[i] : (T)0);
            ext = i == 0 ? x : ext * x;
          }
        }
        acc += prod;
        if constexpr (HVPOI) vol += ext;
      }
    }
    __syncthreads();
  }
  // the G slots of each candidate summed in a fixed order (bit-reproducible); the box stage is free after the loop
  T *red = reinterpret_cast<T *>(bx);
  red[threadIdx.x] = acc;
  if constexpr (HVPOI) red[ACQ_THREADS + threadIdx.x] = vol;
  __syncthreads();
  double val = -INFINITY;
  const bool owner = threadIdx.x < tile && c0 + threadIdx.x < m;
  if (owner) {
    T sum = 0;
    for (int g = 0; g < G; ++g) sum += red[g * tile + threadIdx.x];
    if constexpr (HVPOI) {
      T imp = 0;
      for (int g = 0; g < G; ++g) imp += red[ACQ_THREADS + g * tile + threadIdx.x];
      const double v = (double)sum * (double)imp;
      if (out_acq) out_acq[c0 + threadIdx.x] = v;
      val = isnan(v) ? -INFINITY : v;
    } else if (FEAS) {
      const double v = (double)sum * pof[threadIdx.x];
      if (out_acq) out_acq[c0 + threadIdx.x] = v;
      val = isnan(v) ? -INFINITY : v;
    } else {
      if (out_acq) out_acq[c0 + threadIdx.x] = (double)sum;
      val = isnan(sum) ? -INFINITY : (double)sum;
    }
  }
  // ---- K5: block arg-max ----
  BestPair bb;
  bb.v = val;
  bb.i = owner ? index_base + c0 + threadIdx.x : 0x7fffffffffffffffLL;
  bb = warp_best(bb);
  __shared__ double sv[ACQ_THREADS / 32];
  __shared__ long long si[ACQ_THREADS / 32];
  if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = bb.v; si[threadIdx.x >> 5] = bb.i; }
  __syncthreads();
  if (threadIdx.x < 32) {
    BestPair q;
    q.v = (threadIdx.x < ACQ_THREADS / 32) ? sv[threadIdx.x] : -INFINITY;
    q.i = (threadIdx.x < ACQ_THREADS / 32) ? si[threadIdx.x] : 0x7fffffffffffffffLL;
    q = warp_best(q);
    if (threadIdx.x == 0) { partials[blockIdx.x].value = q.v; partials[blockIdx.x].index = q.i; }
  }
}

// the largest tile whose shared memory leaves room for two CTAs per SM, else the largest that fits at all
template <typename T>
static int box_tile(int k, int B, bool feas) {
  for (int t = 32; t >= 8; t >>= 1) if (box_smem_bytes<T>(k, B, t, feas) <= 110 * 1024) return t;
  return box_smem_bytes<T>(k, B, 8, feas) <= 220 * 1024 ? 8 : 0;    // + the static arg-max slots, under 227 KB
}

template <typename T, int K, int MODE>
static int launch_box(ombo_ctx *ctx, const ombo_acq *acq, int n_gp, const double *mu, const double *var, long long m,
                      long long ld, long long index_base, double *out_acq, cudaStream_t s) {
  constexpr bool FEAS = MODE == BOX_FEAS;
  const int tile = box_tile<T>(K, acq->n_pf, FEAS);
  OMBO_CHECK(tile > 0, "EHVI_BOX: %d breakpoints x %d objectives do not fit in shared memory", acq->n_pf, K);
  const size_t smem = box_smem_bytes<T>(K, acq->n_pf, tile, FEAS);
  if (smem > 48 * 1024)
    OMBO_CUDA(cudaFuncSetAttribute(k_acquire_box<T, K, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long blocks = (m + tile - 1) / tile;
  int rc = ombo_ws_reserve(&ctx->ws_partial, &ctx->ws_partial_bytes, (size_t)blocks * sizeof(ombo_best));
  if (rc) return rc;
  k_acquire_box<T, K, MODE><<<(unsigned)blocks, ACQ_THREADS, smem, s>>>(*acq, tile, mu, var, m, ld, index_base,
                                                                        (const uint4 *)ctx->ws_box, out_acq,
                                                                        (ombo_best *)ctx->ws_partial, n_gp);
  ctx->launches += 1;
  return (int)blocks;
}

template <int MODE>
static int launch_box_k(ombo_ctx *ctx, const ombo_acq *acq, int n_gp, const double *mu, const double *var,
                        long long m, long long ld, long long index_base, double *out_acq, cudaStream_t s, bool fp32) {
  switch (acq->n_obj) {
    case 2: return fp32 ? launch_box<float, 2, MODE>(ctx, acq, n_gp, mu, var, m, ld, index_base, out_acq, s)
                        : launch_box<double, 2, MODE>(ctx, acq, n_gp, mu, var, m, ld, index_base, out_acq, s);
    case 3: return fp32 ? launch_box<float, 3, MODE>(ctx, acq, n_gp, mu, var, m, ld, index_base, out_acq, s)
                        : launch_box<double, 3, MODE>(ctx, acq, n_gp, mu, var, m, ld, index_base, out_acq, s);
    default: return fp32 ? launch_box<float, 4, MODE>(ctx, acq, n_gp, mu, var, m, ld, index_base, out_acq, s)
                         : launch_box<double, 4, MODE>(ctx, acq, n_gp, mu, var, m, ld, index_base, out_acq, s);
  }
}

// OMBO_ACQ_EHVI_BOX, OMBO_ACQ_EHVI_BOX_FEAS and OMBO_ACQ_HV_POI_BOX
static int ombo_acquire_box(ombo_ctx *ctx, const ombo_acq *acq, int n_gp, const double *mu, const double *var,
                            long long m, long long ld, long long index_base, double *out_acq, ombo_best *best_dev,
                            cudaStream_t s, bool fp32) {
  const int k = acq->n_obj;
  int rc = ombo_ws_reserve(&ctx->ws_box, &ctx->ws_box_bytes, (size_t)acq->n_cells * sizeof(uint4));
  if (rc) return rc;
  k_pack_boxes<<<(acq->n_cells + 255) / 256, 256, 0, s>>>(acq->cells, acq->n_cells, k, acq->n_pf,
                                                          (uint4 *)ctx->ws_box);
  ctx->launches += 1;
  fp32 = fp32 && !ctx->knobs.acq_fp64;
  const int blocks =
      acq->kind == OMBO_ACQ_EHVI_BOX_FEAS ? launch_box_k<BOX_FEAS>(ctx, acq, n_gp, mu, var, m, ld, index_base, out_acq, s, fp32)
      : acq->kind == OMBO_ACQ_HV_POI_BOX  ? launch_box_k<BOX_HVPOI>(ctx, acq, n_gp, mu, var, m, ld, index_base, out_acq, s, fp32)
                                          : launch_box_k<BOX_EHVI>(ctx, acq, n_gp, mu, var, m, ld, index_base, out_acq, s, fp32);
  if (blocks < 0) return blocks;
  if (best_dev) {
    k_argmax_final<<<1, 1024, 0, s>>>((const ombo_best *)ctx->ws_partial, blocks, best_dev);
    ctx->launches += 1;
  }
  OMBO_CUDA(cudaGetLastError());
  return OMBO_OK;
}

int ombo_acquire(ombo_ctx *ctx, const ombo_acq *acq, int n_gp, const double *mu, const double *var,
                 long long m, long long ld, long long index_base, double *out_acq, ombo_best *best_dev,
                 cudaStream_t s, bool fp32) {
  if (m <= 0) return OMBO_OK;
  if (acq->kind == OMBO_ACQ_EHVI_BOX || acq->kind == OMBO_ACQ_EHVI_BOX_FEAS || acq->kind == OMBO_ACQ_HV_POI_BOX)
    return ombo_acquire_box(ctx, acq, n_gp, mu, var, m, ld, index_base, out_acq, best_dev, s, fp32);
  int n_stage = 0;
  if (acq->kind == OMBO_ACQ_EHVI2D) n_stage = 2 * (acq->n_pf + 2);
  else if (acq->kind == OMBO_ACQ_HV_POI) n_stage = acq->n_cells * 2 * acq->n_obj;
  else if (acq->kind == OMBO_ACQ_EHVI3D || acq->kind == OMBO_ACQ_EXPECTED_DECOMP) n_stage = acq->n_samples * acq->n_obj;
  size_t smem = (size_t)n_stage * 8;
  OMBO_CHECK(smem <= 200 * 1024, "acquisition constants (%zu B) exceed shared memory", smem);
  // FP32 arithmetic only in the fast precision mode, and never for the expected decomposition (see k_acquire)
  fp32 = fp32 && acq->kind != OMBO_ACQ_EXPECTED_DECOMP && !ctx->knobs.acq_fp64;
  if (smem > 48 * 1024) {   // per (function, device): set whenever the opt-in is needed
    OMBO_CUDA(cudaFuncSetAttribute(k_acquire<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    OMBO_CUDA(cudaFuncSetAttribute(k_acquire<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  int blocks = (int)((m + ACQ_THREADS - 1) / ACQ_THREADS);
  int rc = ombo_ws_reserve(&ctx->ws_partial, &ctx->ws_partial_bytes, (size_t)blocks * sizeof(ombo_best));
  if (rc) return rc;
  if (fp32)
    k_acquire<float><<<blocks, ACQ_THREADS, smem, s>>>(*acq, n_gp, mu, var, m, ld, index_base, out_acq,
                                                       (ombo_best *)ctx->ws_partial);
  else
    k_acquire<double><<<blocks, ACQ_THREADS, smem, s>>>(*acq, n_gp, mu, var, m, ld, index_base, out_acq,
                                                        (ombo_best *)ctx->ws_partial);
  ctx->launches += 1;
  if (best_dev) {
    k_argmax_final<<<1, 1024, 0, s>>>((const ombo_best *)ctx->ws_partial, blocks, best_dev);
    ctx->launches += 1;
  }
  OMBO_CUDA(cudaGetLastError());
  return OMBO_OK;
}
