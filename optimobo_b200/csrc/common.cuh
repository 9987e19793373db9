// Shared declarations for the optimobo_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>

#include "../../include/optimobo_b200.h"

#define OMBO_NB 64            // Cholesky / triangular-inverse block size
#define OMBO_PAD 128          // n_pad granularity (GEMM N-chunk)
#define OMBO_PROF_MAX 4096
#define OMBO_F8C_KAPPA_DEFAULT 100.0   // conditioning limit of the f8c operand format (measured, DESIGN.md section 4)
#define OMBO_CHUNK (1 << 20)  // candidates per pass of the HOST entry (H2D staging granularity: copy i+1 overlaps pass i)
// device pools: candidates per pass through the posterior workspace (OMBO_CHUNK_LOG2).  A launch of the persistent
// posterior kernels loses about one tile time to fill / drain and up to one tile per CTA to the ragged last wave:
// 2^22 instead of 2^20 candidates per launch takes that from ~3 % to under 1 % of the kernel time at C5.
#define OMBO_CHUNK_DEV_LOG2 22

void ombo_set_error(const char *fmt, ...);

#define OMBO_CUDA(call)                                                              \
  do {                                                                               \
    cudaError_t e__ = (call);                                                        \
    if (e__ != cudaSuccess) {                                                        \
      ombo_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,                   \
                     cudaGetErrorString(e__));                                       \
      return OMBO_ERR_CUDA;                                                          \
    }                                                                                \
  } while (0)

#define OMBO_CHECK(cond, ...)                                                        \
  do {                                                                               \
    if (!(cond)) {                                                                   \
      ombo_set_error(__VA_ARGS__);                                                   \
      return OMBO_ERR_INVALID;                                                       \
    }                                                                                \
  } while (0)

// environment knobs, read ONCE when the context is created (never on the launch path)
struct ombo_knobs {
  int fast_dbg;           // OMBO_FAST_DBG: timing experiments (results are garbage)
  int fast_profile;       // OMBO_FAST_PROFILE: per-CTA wait-cycle counters printed to stderr
  int fast_gen_warps;     // OMBO_FAST_GEN_WARPS: 8 or 16 K1 generator warps in the f8c kernel (0: 8, bound launches 16)
  int f8_max_run;         // OMBO_F8_MAXRUN: most reload steps in a row between two generated blocks
  double f8_tg;           // OMBO_F8_TG: generator time per K-block in units of one 256-column MMA unit (schedule)
  int chunk_log2;         // OMBO_CHUNK_LOG2: device-pool candidates per pass = 2^chunk_log2
  int no_f8c;             // OMBO_NO_F8C: never choose the fp16 + 2 x e4m3 operand format
  double f8c_kappa;       // OMBO_F8C_KAPPA: conditioning limit of that format
  int acq_fp64;           // OMBO_ACQ_FP64: keep the FP64 acquisition kernel in fast mode
  int no_fuse;            // OMBO_NO_FUSE: never fuse the 2-D EHVI + arg-max into the f8c kernel's epilogue
  int no_prune;           // OMBO_NO_PRUNE: score every candidate in full even where a variance bound could skip most
  int prune_depth;        // OMBO_PRUNE_DEPTH: 256-column chunks of V behind the variance bound (1 or 2)
  long long prune_cap;    // OMBO_PRUNE_CAP: most survivors scored in full before falling back (0: max(2^16, m / 64))
  int prune_log;          // OMBO_PRUNE_LOG: one stderr line per pruned call (survivors, bound, threshold)
  int prune_stage1;       // OMBO_PRUNE_STAGE1=0: no mean-only first stage in front of the variance bound
  long long prune_cap1;   // OMBO_PRUNE_STAGE1_CAP: most stage-1 survivors before the depth-1 path takes the whole pool
                          //   (0: max(2^16, m / 8))
  int stage1_mean8;       // OMBO_STAGE1_KERNEL=mean8: stage 1 on k_posterior_mean8 even where the tensor-core kernel covers
};

struct ombo_ctx {
  int device;
  int num_sms;
  int64_t launches;
  ombo_knobs knobs;
  long long *prof_dev;    // per-CTA wait counters of the fast kernels (OMBO_FAST_PROFILE)
  // step schedules of the f8c kernel (posterior_fast8.cu), [0] full, [1] bound; rebuilt when n_pad or the depth changes
  unsigned int *f8_sched[2]; int f8_sched_np[2], f8_sched_depth[2], f8_sched_len[2], f8_sched_cap[2];
  // workspaces (grown on demand, freed in ctx_destroy)
  void *ws_post;      size_t ws_post_bytes;      // posterior mu/var chunk buffers
  void *ws_scratch;   size_t ws_scratch_bytes;   // FP64 K* tiles (L2 resident) / fast-path scratch
  void *ws_partial;   size_t ws_partial_bytes;   // per-block arg-max partials
  void *ws_box;       size_t ws_box_bytes;       // EHVI_BOX boxes as packed 16-bit breakpoint indices
  void *ws_prune;     size_t ws_prune_bytes;     // pruned scoring: per-candidate upper bounds, survivors, cub scratch
  void *ws_prune1;    size_t ws_prune1_bytes;    // its mean-only first stage: bounds, survivors and their rows
  void *ws_topk;      size_t ws_topk_bytes;      // top-k: one pass's keys, the running k-list, selections, cub scratch
  void *ws_boxprep;   size_t ws_boxprep_bytes;   // ombo_ehvi_boxes: flags, ranks, slice lists, tuples, counts, table
  void *ws_stage[2];  size_t ws_stage_bytes;     // host-entry H2D staging (double buffered)
  void *ws_best;                                  // 16 B device best for the host entry
  ombo_best *pinned_best;                         // pinned host landing zone
  cudaStream_t copy_stream;
  cudaEvent_t ev_copied[2], ev_consumed[2];
  // optional per-launch timing of the posterior kernels
  int prof_enabled;
  int prof_count;
  cudaEvent_t prof_ev[2 * OMBO_PROF_MAX];
};

// brackets one posterior-kernel launch with events when profiling is on
struct ProfScope {
  ombo_ctx *c; cudaStream_t s; int slot;
  ProfScope(ombo_ctx *ctx, cudaStream_t st) : c(ctx), s(st), slot(-1) {
    if (c->prof_enabled && c->prof_count < OMBO_PROF_MAX) {
      slot = c->prof_count++;
      cudaEventRecord(c->prof_ev[2 * slot], s);
    }
  }
  ~ProfScope() { if (slot >= 0) cudaEventRecord(c->prof_ev[2 * slot + 1], s); }
};

int ombo_ws_reserve(void **p, size_t *cur, size_t want);

// ---- state blob layout: a pure function of (n, d) -----------------------------------
struct GpLayout {
  int n, d, n_pad;
  size_t off_L, off_Linv, off_alpha, off_xs, off_status, off_dinv, off_tmp, off_inv_ell;
  size_t off_bhi, off_blo, off_xs32, off_alpha32, off_center, off_b2, off_bscale;
  size_t bytes;
};

static inline int ombo_round_up(int x, int q) { return (x + q - 1) / q * q; }

static inline GpLayout gp_layout(int n, int d) {
  GpLayout L;
  L.n = n; L.d = d; L.n_pad = ombo_round_up(n < 1 ? 1 : n, OMBO_PAD);
  size_t np = (size_t)L.n_pad, off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  L.off_L = take(np * np * 8);
  L.off_Linv = take(np * np * 8);
  L.off_alpha = take(np * 8);
  L.off_xs = take((size_t)d * np * 8);
  L.off_status = take(16);
  L.off_dinv = take((np / OMBO_NB) * OMBO_NB * OMBO_NB * 8);
  L.off_tmp = take(np * 8);
  L.off_inv_ell = take((size_t)OMBO_MAX_DIM * 8);
  L.off_bhi = take(np * np * 2);
  L.off_blo = take(np * np * 2);
  L.off_xs32 = take(np * 32 * 4);
  L.off_alpha32 = take(np * 4);
  L.off_center = take((size_t)OMBO_MAX_DIM * 8);
  L.off_b2 = take(np * 4);
  L.off_bscale = take(32);                // after the refresh: [1] scale s of the 16-bit planes, [2] 1/s^2, [3] 1.0 = fp16 / 0.0 = bf16
  L.bytes = off;
  return L;
}

// device-side view of one GP used by the scoring kernels
struct GpDev {
  int n, n_pad, d, kernel;
  int flags;              // ombo_gp.reserved: bit 0 = OMBO_GP_DIRECT_DISTANCES (fast mode)
  double sigma_f2, sigma_n2, var_floor;
  const double *xs;       // (d, n_pad) scaled
  const double *ell;      // (d) length-scales
  const double *Linv;     // (n_pad, n_pad)
  const double *alpha;    // (n_pad)
  const unsigned short *bhi, *blo;       // 16-bit hi / lo planes of s * sigma_f2 * L^-1 (bf16 or fp16, see bscale[3])
  const double *bscale;                  // [1] = s, [2] = 1 / s^2 (power of two: exact), [3] = 1.0 fp16 / 0.0 bf16
  const float *xs32, *alpha32, *b2_32;   // fast path: centred scaled inputs, sigma_f2*alpha, |xs32_i|^2
  const double *center;                  // (d) per-dimension mean of the training inputs
};

static inline GpDev gp_dev_view(const ombo_gp &g) {
  GpLayout L = gp_layout(g.n, g.d);
  const char *b = (const char *)g.state;
  GpDev v;
  v.n = g.n; v.n_pad = L.n_pad; v.d = g.d; v.kernel = g.kernel; v.flags = g.reserved;
  v.sigma_f2 = g.sigma_f2; v.sigma_n2 = g.sigma_n2; v.var_floor = g.var_floor;
  v.xs = (const double *)(b + L.off_xs);
  v.ell = (const double *)(b + L.off_inv_ell);
  v.Linv = (const double *)(b + L.off_Linv);
  v.alpha = (const double *)(b + L.off_alpha);
  v.bhi = (const unsigned short *)(b + L.off_bhi);
  v.blo = (const unsigned short *)(b + L.off_blo);
  v.bscale = (const double *)(b + L.off_bscale);
  v.xs32 = (const float *)(b + L.off_xs32);
  v.alpha32 = (const float *)(b + L.off_alpha32);
  v.b2_32 = (const float *)(b + L.off_b2);
  v.center = (const double *)(b + L.off_center);
  return v;
}

// candidate pool as the kernels see it
struct PoolDev {
  const void *X;      // device rows for this pass (already offset), or nullptr
  int dtype, d;
  long long index_base;   // global index of local row 0 of this pass
  unsigned long long seed;
  double lo[OMBO_MAX_DIM], span[OMBO_MAX_DIM];
};

// f8c kernel: 2-D EHVI and the per-CTA arg-max evaluated by the epilogue warps of the last launch of a pass (K4 + K5
// fused behind K2: that model's mu / var never leave the SM, the other model's come from the posterior workspace).
// Exact semantics: model 0 first, model 1 carries the acquisition.  Reference semantics reads only model 0's variance
// (util_functions.py:233), so model 1 runs first in the mean-only kernel and model 0's launch carries it.
struct FuseAcq {
  int on;                      // 0: plain posterior launch (mu_out / var_out written)
  int n_pf, exact;             // stripes y1[0..P+1], y2[0..P+1]; semantics flag of ehvi2d_value
  float c00, c01;              // reference semantics: flattened sample covariance entries
  int self_model;              // which objective this launch computes (0 or 1)
  const double *mu_other, *var_other;   // posterior of the other model for the same candidates (var_other may be NULL)
  const double *stripes;       // device, 2 (P + 2) doubles
  double *out_acq;             // optional per-candidate values
  ombo_best *partials;         // [gridDim.x] per-CTA (value, global index)
  long long index_base;        // global index of candidate 0 of this launch
};

// ---- internal entry points (one per .cu) ------------------------------------------------
// api.cu: the argument checks of every scoring entry, and one pass of it: rows [first, first + count) of the pool,
// X_dev pointing at row `first` (NULL: generator); out_mu / out_var / out_acq are offset by `first`
int ombo_validate_score(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const ombo_acq *acq,
                        int precision);
int ombo_score_pass(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const void *X_dev,
                    long long first, long long count, const ombo_acq *acq, int precision, double *out_mu,
                    double *out_var, double *out_acq, long long out_ld, ombo_best *best_dev, cudaStream_t s,
                    int bound_chunks = 0);
int ombo_refresh_impl(ombo_ctx *ctx, const ombo_gp_spec *spec, void *state, cudaStream_t s);
int ombo_nlml_grad_impl(ombo_ctx *ctx, const ombo_gp_spec *spec, void *state, double *out_host, cudaStream_t s);
int ombo_posterior_fp64(ombo_ctx *ctx, const GpDev &gp, const PoolDev &pool, long long m,
                        double *mu, double *var, bool want_var, cudaStream_t s);
// fuse_req != NULL asks for the fused 2-D EHVI + arg-max epilogue; *fused reports whether the launch did it (only
// the f8c kernel can, and only while the stripes fit beside its operand rings) -- if not, mu / var were written
// and the caller runs K4 as usual
// bound_chunks >= 1 (f8c planes only): var is the upper bound from the first bound_chunks 256-column chunks of V
// (posterior_fast8.cu, BOUND schedule), mu and everything else as in a full launch
int ombo_posterior_fast(ombo_ctx *ctx, const GpDev &gp, const PoolDev &pool, long long m,
                        double *mu, double *var, bool want_var, cudaStream_t s,
                        const FuseAcq *fuse_req = nullptr, int *fused = nullptr, int bound_chunks = 0);
int ombo_posterior_fast8(ombo_ctx *ctx, const GpDev &gp, const PoolDev &pool, long long m,
                         double *mu, double *var, cudaStream_t s,
                         const FuseAcq *fuse_req = nullptr, int *fused = nullptr, int bound_chunks = 0);
// whether an f8c launch for this GP can carry the fused 2-D EHVI of a front of n_pf points (shared memory)
bool ombo_f8_can_fuse(ombo_ctx *ctx, const GpDev &gp, int n_pf, int bound_chunks, cudaStream_t s);
// posterior_mean8.cu: stage 1 of the pruned arg-max, the mean-only bound of the exact 2-D EHVI of an f8c pair for every
// candidate of a pool (ub[m], mu_out [2][m] optional) and the largest into *best_dev; covers d <= 12 while both
// training sets fit in shared memory.  *grid_out (optional): the CTAs launched, whose per-CTA maxima are left in
// ctx->ws_partial
bool ombo_mean8_covers(const GpDev gp[2], int n_pf);
int ombo_mean8_bound(ombo_ctx *ctx, const GpDev gp[2], const PoolDev &pool, long long m, const double *stripes,
                     int n_pf, float c00, float c01, double *ub, ombo_best *best_dev, double *mu_out, int *grid_out,
                     cudaStream_t s);
// posterior_stage1_tc.cu: the same bound with tcgen05 distances and a certified margin on each mean (the default stage
// 1 where it covers the shape: d <= 12, both training sets' fp16 planes in shared memory); mu_out / marg_out
// (optional, [2][m] each): the stage-1 means and their margins
bool ombo_stage1_tc_covers(const GpDev gp[2], int n_pf);
// whether its margin stays small enough to prune well for this pool (the largest a2 and |b|^2 of both GPs, from the
// pool's box or a scan; ws: 32 bytes of device workspace; one stream synchronise)
int ombo_stage1_tc_useful(ombo_ctx *ctx, const GpDev gp[2], const PoolDev &pool, long long m, void *ws, bool *useful,
                          cudaStream_t s);
int ombo_stage1_tc_bound(ombo_ctx *ctx, const GpDev gp[2], const PoolDev &pool, long long m, const double *stripes,
                         int n_pf, float c00, float c01, double *ub, ombo_best *best_dev, double *mu_out,
                         double *marg_out, int *grid_out, cudaStream_t s);
// merges n_partials per-block (value, index) pairs in ctx->ws_partial with the running best
int ombo_argmax_merge(ombo_ctx *ctx, int n_partials, ombo_best *best_dev, cudaStream_t s);
int ombo_fast_path_built();
int ombo_acquire(ombo_ctx *ctx, const ombo_acq *acq, int n_gp, const double *mu, const double *var,
                 long long m, long long ld, long long index_base, double *out_acq,
                 ombo_best *best_dev, cudaStream_t s, bool fp32 = false);
int ombo_scalarise_impl(ombo_ctx *ctx, const ombo_acq *acq, const double *F, long long m, double *out, cudaStream_t s);
int ombo_best_init(ombo_ctx *ctx, ombo_best *best_dev, cudaStream_t s);
int ombo_pack_key_impl(ombo_ctx *ctx, const ombo_best *best_dev, long long *key_dev, cudaStream_t s);
int ombo_potrf_lower_impl(ombo_ctx *ctx, double *L, int np, int n, double *dinv, int *status, cudaStream_t s);
// posterior_joint.cu (SURVEY section 8f rank 4)
int ombo_joint_samples_impl(ombo_ctx *ctx, const ombo_gp &g, const double *Xc, int m, const double *Z, int S,
                            double diag_add, double *out, cudaStream_t s);
// front_prep.cu (SURVEY section 8f rank 2)
int ombo_pareto_mask_impl(ombo_ctx *ctx, const double *Y, int n, int k, unsigned char *mask, cudaStream_t s);
int ombo_hypervolume_impl(ombo_ctx *ctx, const double *P, int p, int k, const double *ref, double *out, cudaStream_t s);
int ombo_cells_2d_impl(ombo_ctx *ctx, const double *PF, int p, const double *ideal, const double *maxp, double *cells,
                       cudaStream_t s);
// box_prep.cu: the box decomposition of host_prep.ehvi_boxes (one synchronise)
int ombo_ehvi_boxes_impl(ombo_ctx *ctx, const double *PF, int p, int k, const double *ref, double *table,
                         double *boxes, long long boxes_cap, int *B_out, long long *n_boxes_out, cudaStream_t s);
int ombo_pool_rows_impl(ombo_ctx *ctx, const PoolDev &pool, long long first, long long count,
                        double *out, cudaStream_t s);
