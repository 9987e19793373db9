/*
 * optimobo_b200 -- C ABI of the B200-native acquisition hot path.
 *
 * The reference (aje220/OptiMOBO) is duck-typed Python with no FFI of its own
 * (SURVEY.md section 8b), so each entry point cites the reference call it replaces:
 *
 *   ombo_gp_refresh   <- GPy.models.GPRegression(X, y, Matern52(ARD)) state build after
 *                        .optimize(): optimobo/algorithms/optimisers.py:226-231, :447-451,
 *                        :494-496; parego.py:217-219; keep.py:220-222,235-237; emo.py:297-300;
 *                        cparego.py:371-373,828-830,837-839            (SURVEY row a14 / K3)
 *   ombo_score        <- the inner-optimiser call site that evaluates the acquisition one x
 *                        at a time: differential_evolution(obj, bounds) at optimisers.py:87,
 *                        :118,:366; cparego.py:94,:544; emo.py:240; the EA loops
 *                        parego.py:242-270, keep.py:260-292       (rows a1-a12 / K1,K2,K4,K5)
 *   ombo_score_host   <- same, with the candidate pool in HOST memory (end-to-end entry)
 *   acquisition kinds <- util_functions.py:136 (EHVI), :170 (EHVI_3D), :285
 *                        (expected_decomposition), optimisers.py:325 / parego.py:126 /
 *                        keep.py:118 / cparego.py:450 (EI), cparego.py:486 (consraint_ei),
 *                        keep.py:142 (pareto_expected_improvement), emo.py:192
 *                        (hypervolume_based_PoI)
 *   scalarisation ids <- optimobo/scalarisations.py:37,53,76,113,153,177,201,222,242,277,314,355
 *
 * Conventions: every function returns an int status (0 = ok, negative = error; the message
 * is available from ombo_last_error()).  All device buffers are owned by the caller
 * (torch tensors) and only borrowed for the call.  `stream` is a cudaStream_t passed as
 * void*.  Nothing here takes or returns a torch type.  One ctx per device / thread.
 */
#ifndef OPTIMOBO_B200_H
#define OPTIMOBO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OMBO_ABI_VERSION 1

#define OMBO_OK               0
#define OMBO_ERR_INVALID     -1
#define OMBO_ERR_NOT_PD      -2   /* K + (sigma_n2 + jitter) I not positive definite */
#define OMBO_ERR_CUDA        -3
#define OMBO_ERR_UNSUPPORTED -4

#define OMBO_MAX_GP   8
#define OMBO_MAX_OBJ  4
#define OMBO_MAX_DIM  32
#define OMBO_MAX_TRAIN 8192

enum { OMBO_KERNEL_MATERN52 = 0, OMBO_KERNEL_RBF = 1 };
enum { OMBO_PREC_FP64 = 0,   /* FP64 DMMA path, reference-tolerance mode (rtol 1e-6)    */
       OMBO_PREC_FAST = 1 }; /* 16-bit x3 split on tcgen05 tensor cores (rtol 1e-3)     */
enum { OMBO_SEM_REFERENCE = 0, /* reproduces the reference's formulas incl. quirks       */
       OMBO_SEM_EXACT = 1 };   /* each model's own sigma, n+1 EHVI stripes               */

enum {
  OMBO_ACQ_NONE = 0,            /* posterior only                                         */
  OMBO_ACQ_EHVI2D = 1,          /* util_functions.py:136-167 + :81-133                    */
  OMBO_ACQ_EHVI3D = 2,          /* util_functions.py:170-214                              */
  OMBO_ACQ_EXPECTED_DECOMP = 3, /* util_functions.py:285-327                              */
  OMBO_ACQ_EI = 4,              /* optimisers.py:325-344 and its four copies              */
  OMBO_ACQ_CONSTRAINED_EI = 5,  /* cparego.py:486-496                                     */
  OMBO_ACQ_PARETO_EI = 6,       /* keep.py:142-150 (gp 0 = pareto model, gp 1 = scalar)   */
  OMBO_ACQ_HV_POI = 7,          /* emo.py:192-228                                         */
  OMBO_ACQ_EHVI_BOX = 8         /* exact EHVI, 2 <= n_obj <= 4, by box decomposition      */
};

/* OMBO_ACQ_EHVI_BOX: the exact expected hypervolume improvement for k = n_obj independent Gaussian objectives,
 *   EHVI = sum_c prod_i (H_i(u_ci) - H_i(l_ci)),  H_i(t) = E[(t - y_i)^+] (H_i(-inf) = 0),
 * over disjoint boxes [l_c, u_c] that tile the part of [-inf, ref] no front point dominates
 * (host_prep.ehvi_boxes builds both tables).  It reuses the fields of ombo_acq:
 *   n_obj   = k                      ref   = the reference point r
 *   n_pf    = B, breakpoints per objective
 *   stripes = DEVICE (k, B) f64: row i = -inf, the sorted distinct front coordinates of objective i, r_i,
 *             padded with r_i to B
 *   cells   = DEVICE (n_cells, 2, k) f64 holding integer breakpoint indices: [c][0] upper, [c][1] lower corner,
 *             index 0 = -inf
 * Each model's own variance is used (semantics is ignored).  Limits: 2 <= B <= OMBO_EHVI_BOX_MAX_BREAKS,
 * 1 <= n_cells <= OMBO_EHVI_BOX_MAX_BOXES; indices outside [0, B) are clamped. */
#define OMBO_EHVI_BOX_MAX_BREAKS 514        /* a front of up to 512 points */
#define OMBO_EHVI_BOX_MAX_BOXES  (1 << 20)

enum {
  OMBO_SC_WEIGHTED_SUM = 0, OMBO_SC_TCHEBICHEFF = 1, OMBO_SC_AUG_TCHEBICHEFF = 2,
  OMBO_SC_MOD_TCHEBICHEFF = 3, OMBO_SC_EXP_WEIGHTED = 4, OMBO_SC_WEIGHTED_NORM = 5,
  OMBO_SC_WEIGHTED_POWER = 6, OMBO_SC_WEIGHTED_PRODUCT = 7, OMBO_SC_PBI = 8,
  OMBO_SC_IPBI = 9, OMBO_SC_QPBI = 10, OMBO_SC_APD = 11
};

typedef struct ombo_ctx ombo_ctx;

/* ---- K3: GP refresh ------------------------------------------------------- */
typedef struct {
  int32_t n, d;             /* training rows, input dimension (d <= OMBO_MAX_DIM)         */
  int32_t kernel;           /* OMBO_KERNEL_*                                              */
  int32_t reserved;
  double sigma_f2;          /* kernel variance                                            */
  double sigma_n2;          /* Gaussian noise variance (reference fixes it to 0)          */
  double jitter;            /* GPy adds 1e-8 to the diagonal                              */
  const double *X;          /* DEVICE (n, d) row-major                                    */
  const double *y;          /* DEVICE (n,)                                                */
  const double *ell;        /* HOST   (d,) ARD length-scales                              */
} ombo_gp_spec;

/* fields of the opaque, caller-owned state blob (offsets via ombo_gp_state_field) */
enum { OMBO_FIELD_L = 0,      /* (n_pad, n_pad) f64 lower Cholesky factor                 */
       OMBO_FIELD_LINV = 1,   /* (n_pad, n_pad) f64 lower-triangular inverse              */
       OMBO_FIELD_ALPHA = 2,  /* (n_pad,) f64                                             */
       OMBO_FIELD_XS = 3,     /* (d, n_pad) f64 length-scale-scaled training inputs       */
       OMBO_FIELD_STATUS = 4, /* (4,) i32: [0] = first non-PD pivot row + 1, 0 if PD       */
       OMBO_FIELD_BHI = 5,    /* (n_pad, n_pad) bf16 | fp16, hi plane of s*sigma_f2*Linv   */
       OMBO_FIELD_BLO = 6,    /* (n_pad, n_pad) lo plane (format / scale chosen by K3)     */
       OMBO_FIELD_XS32 = 7,   /* (32, n_pad) f32 centred scaled training inputs (fast path) */
       OMBO_FIELD_ALPHA32 = 8 /* (n_pad,) f32 alpha * sigma_f2                              */
};

int ombo_abi_version(void);
int ombo_has_fast_path(void);   /* 1 when OMBO_PREC_FAST (tcgen05) is compiled in */
const char *ombo_last_error(void);

int ombo_ctx_create(int device, ombo_ctx **out);
int ombo_ctx_destroy(ombo_ctx *ctx);

int ombo_n_pad(int n);
int ombo_gp_state_bytes(int n, int d, size_t *bytes);
int ombo_gp_state_field(int n, int d, int field, size_t *byte_offset, size_t *n_elems);

/* Builds K, L = chol(K + (sigma_n2 + jitter) I), L^-1, alpha (+ fast-path planes) into
 * `state` (device, ombo_gp_state_bytes).  Synchronises `stream` once at the end to read the
 * PD status: returns OMBO_ERR_NOT_PD so the host can raise the jitter and retry (GPy jitchol). */
int ombo_gp_refresh(ombo_ctx *ctx, const ombo_gp_spec *spec, void *state, void *stream);

/* Hyper-parameter fit support (SURVEY section 8f-1): refreshes `state` for the hyper-parameters in `spec`
 * and returns on the HOST out[0] = negative log marginal likelihood, out[1] = d/d log sigma_f2,
 * out[2 + j] = d/d log ell_j (d + 2 doubles).  Replaces the O(n^3) work inside GPy's
 * model.optimize(max_f_eval=1000) (optimisers.py:230 ...); the L-BFGS driver stays on the host.
 * Synchronises `stream`.  OMBO_ERR_NOT_PD as for ombo_gp_refresh. */
int ombo_gp_nlml_grad(ombo_ctx *ctx, const ombo_gp_spec *spec, void *state, double *out_host, void *stream);

/* ---- scoring --------------------------------------------------------------- */
/* ombo_gp.reserved carries the flags of the refreshed state.  ombo_gp_refresh chooses the format of the fast
 * mode's operand planes on the device from the conditioning of the Cholesky factor -- bf16 (well conditioned) or
 * scaled fp16 together with direct-difference distances (ill conditioned, DESIGN.md) -- and reports it in
 * OMBO_FIELD_STATUS word 1 of the state blob (1 = fp16).  The caller copies it into bit 1 of `reserved`;
 * the scoring entries launch the matching kernel instantiation.  fp16 planes are only produced when the refresh
 * was asked for them (ombo_gp_spec.reserved bit 1 set): a caller that leaves both `reserved` fields 0 always
 * gets, and scores with, bf16 planes. */
#define OMBO_GP_FP16_PLANES 2
/* Third format, "f8c" (status word 1 = 2, bit 2 of `reserved`): hi plane fp16, lo field = two e4m3 planes
 * (e4m3(2^-12 B) and e4m3(B - fp16(B))) for the pair kernel that runs one fp16 product plus two e4m3 correction
 * products (2.0 tensor units per MAC instead of 3.0).  Chosen only when the refresh was asked for it (spec bit 2),
 * d <= 12 and the conditioning proxy is below the measured limit (DESIGN.md section 4). */
#define OMBO_GP_F8C_PLANES 4
typedef struct {
  int32_t n, d, kernel, reserved;
  double sigma_f2, sigma_n2;
  double var_floor;          /* GPy clips the variance at 1e-15; sklearn surface: 0        */
  const void *state;         /* DEVICE blob filled by ombo_gp_refresh                      */
} ombo_gp;

typedef struct {
  const void *X;             /* (m, d) row-major candidates, or NULL: counter-generated    */
  int32_t dtype;             /* 0 = f64, 1 = f32                                           */
  int32_t d;
  int64_t m;
  int64_t index_base;        /* global index of row 0 (shards of one pool on several GPUs) */
  uint64_t seed;             /* generator key                                              */
  double lo[OMBO_MAX_DIM];   /* generator box                                              */
  double hi[OMBO_MAX_DIM];
} ombo_pool;

typedef struct {
  int32_t kind;              /* OMBO_ACQ_*                                                 */
  int32_t semantics;         /* OMBO_SEM_*                                                 */
  int32_t scalarisation;     /* OMBO_SC_* (EXPECTED_DECOMP)                                */
  int32_t n_obj;
  int32_t n_pf;              /* EHVI2D: |PF| = P (stripes holds 2*(P+2) doubles)           */
  int32_t n_cells;           /* HV_POI                                                     */
  int32_t n_samples;         /* S, rows of cache                                           */
  int32_t reserved;
  double best;               /* EI family: current best; EXPECTED_DECOMP: g_min; EHVI3D: HV(PF) */
  double var_eps[OMBO_MAX_GP]; /* added to var before sqrt (0, 1e-6, 1e-5: SURVEY a8,a9,a11) */
  double ref[OMBO_MAX_OBJ];  /* reference / max point                                      */
  double ideal[OMBO_MAX_OBJ], maxp[OMBO_MAX_OBJ], weights[OMBO_MAX_OBJ];
  double sc_params[4];       /* alpha|p|theta, alpha, H / FE, FE_max, gamma                */
  double cache_c00, cache_c01; /* np.cov(cache[:,0], cache[:,1]) entries (EHVI reference)  */
  const double *stripes;     /* DEVICE (2, P+2): y1 then y2, util_functions.py:94-112      */
  const double *cells;       /* DEVICE (n_cells, 2, n_obj): [c][0] upper, [c][1] lower      */
  const double *cache;       /* DEVICE (S, n_obj)                                          */
} ombo_acq;

typedef struct { double value; int64_t index; } ombo_best;   /* 16 bytes */

/* K1+K2 (+K4+K5): scores pool->m candidates.  Optional DEVICE outputs: out_mu/out_var
 * (n_gp, m) f64, out_acq (m,) f64, best (16 B; max acquisition, ties -> lowest global index,
 * NaN treated as -inf).  Asynchronous on `stream`. */
int ombo_score(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool,
               const ombo_acq *acq, int precision, double *out_mu, double *out_var,
               double *out_acq, ombo_best *best_dev, void *stream);

/* End-to-end twin: pool->X is a HOST buffer (pinned for full speed); chunks are copied
 * host->device on a side stream overlapped with scoring; `best_host` is read back and the
 * call returns after the result is on the host. */
int ombo_score_host(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool,
                    const ombo_acq *acq, int precision, ombo_best *best_host, void *stream);

/* The device scalarisation switch on explicit objective vectors: out[r] = g(F[r, :], weights) with F DEVICE (m, n_obj)
 * row-major f64 and the function / bounds / weights / parameters taken from `acq` (scalarisation, n_obj, ideal, maxp,
 * weights, sc_params).  Device twin of `Scalarisation.__call__(F, weights)` (optimobo/scalarisations.py:20-27, the
 * twelve `_do` at :43,66,92,130,165,190,212,230,257,291,325,375); checked against the reference-minted fixtures. */
int ombo_scalarise(ombo_ctx *ctx, const ombo_acq *acq, const double *F, int64_t m, double *out, void *stream);

/* K4+K5 alone on caller-supplied posteriors: mu/var DEVICE (n_gp, ld) f64, m <= ld candidates.
 * Lets the acquisition arithmetic be checked against fixtures independently of the GP path. */
int ombo_acquire_posterior(ombo_ctx *ctx, const ombo_acq *acq, int n_gp, const double *mu,
                           const double *var, int64_t m, int64_t ld, int64_t index_base,
                           double *out_acq, ombo_best *best_dev, void *stream);

/* regenerates rows [index, index+count) of a counter-generated pool into DEVICE out (count,d) f64 */
int ombo_pool_rows(ombo_ctx *ctx, const ombo_pool *pool, int64_t index, int64_t count,
                   double *out, void *stream);

/* C1 support: packs the 16-byte best into ONE order-preserving signed 64-bit key for a single
 * NCCL all-reduce(MAX): high 32 bits = order-preserving image of (float)value, low 32 bits =
 * 0xFFFFFFFF - global index (so ties resolve to the lowest index, like np.argmax).  key_dev is
 * DEVICE int64; it can be the NCCL send buffer itself.  Requires 0 <= index < 2^32. */
int ombo_pack_key(ombo_ctx *ctx, const ombo_best *best_dev, int64_t *key_dev, void *stream);

/* ---- candidate-independent prep on the device (SURVEY.md section 8f rank 2) ----------------------
 * Replaces the reference's pygmo / pymoo calls of every BO iteration; all pointers are DEVICE float64
 * row-major unless noted, results are bit-identical to optimobo_b200/host_prep.py.
 *
 * ombo_pareto_mask: mask[j] = 1 iff row j of Y (n,k) is in the first non-dominated front (minimisation;
 *   pygmo.fast_non_dominated_sorting(...)[0][0], util_functions.py:64-77).  1 <= k <= 8.
 * ombo_hypervolume: exact dominated hypervolume of P (p,k), k = 2 or 3, w.r.t. ref (HOST, k doubles);
 *   points beyond ref contribute nothing (pymoo HV optimisers.py:217-219; pygmo hypervolume.compute
 *   util_functions.py:198-199).  hv_out: DEVICE double[1].  p <= 16384.
 * ombo_cells_2d: the (p+1, 2, 2) cell decomposition of a 2-D front EMO scores against
 *   (emo.py:55-152): [c][0] = upper, [c][1] = lower corner.  ideal / maxp: HOST double[2].  p >= 1. */
int ombo_pareto_mask(ombo_ctx *ctx, const double *Y, int n, int k, unsigned char *mask, void *stream);
int ombo_hypervolume(ombo_ctx *ctx, const double *P, int p, int k, const double *ref, double *hv_out,
                     void *stream);
int ombo_cells_2d(ombo_ctx *ctx, const double *PF, int p, const double *ideal, const double *maxp,
                  double *cells, void *stream);

/* ---- joint posterior samples (SURVEY.md section 8f rank 4) --------------------------------------------
 * The device side of TuRBO's Thompson sampling, `GP.posterior_samples(X_cand, size=batch_size)`
 * (turbo.py:75-117): out = mu + chol(K** - K*^T Ky^-1 K* + diag_add I) Z for the m candidates Xc (DEVICE f64
 * (m,d) row-major), Z = DEVICE f64 (m,S) standard normals supplied by the caller, out DEVICE f64 (m,S).
 * diag_add = likelihood noise + jitter.  FP64 throughout.  1 <= m <= 16384, S >= 1.  Returns OMBO_ERR_NOT_PD
 * when the posterior covariance is not numerically positive definite (raise diag_add and retry).
 * Synchronises the stream (status readback). */
int ombo_posterior_joint_samples(ombo_ctx *ctx, const ombo_gp *gp, const double *Xc, int m, const double *Z,
                                 int n_samples, double diag_add, double *out, void *stream);

/* Per-kernel timing of the dominant (posterior) kernel with CUDA events recorded on the
 * launching stream: enable, run, synchronise, then read the launch count and total duration. */
int ombo_profile_enable(ombo_ctx *ctx, int enable);
int ombo_profile_read(ombo_ctx *ctx, int64_t *n_launches, double *total_ms);

/* number of kernels this library launched since the counter was last reset (bench.py's
 * gpu_launches) */
int64_t ombo_launch_count(ombo_ctx *ctx, int reset);

#ifdef __cplusplus
}
#endif
#endif
