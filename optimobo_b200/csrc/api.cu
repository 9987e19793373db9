// C-ABI entry points (include/optimobo_b200.h).  Plain pointers and sizes only.
#include <stdarg.h>
#include <stdlib.h>

#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "acq_math.cuh"
#include "candidates.cuh"

static thread_local char g_err[1024] = "";

void ombo_set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int ombo_ws_reserve(void **p, size_t *cur, size_t want) {
  if (*cur >= want && *p) return OMBO_OK;
  if (*p) {
    OMBO_CUDA(cudaDeviceSynchronize());
    OMBO_CUDA(cudaFree(*p));
    *p = nullptr; *cur = 0;
  }
  size_t bytes = (want + (1 << 20) - 1) / (1 << 20) * (1 << 20);
  OMBO_CUDA(cudaMalloc(p, bytes));
  *cur = bytes;
  return OMBO_OK;
}

extern "C" {

int ombo_abi_version(void) { return OMBO_ABI_VERSION; }
int ombo_has_fast_path(void) { return ombo_fast_path_built(); }
const char *ombo_last_error(void) { return g_err; }

int ombo_ctx_create(int device, ombo_ctx **out) {
  OMBO_CHECK(out != nullptr, "ctx_create: out is NULL");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    ombo_set_error("ctx_create: no CUDA device (%s) -- optimobo_b200 has no CPU fallback",
                   cudaGetErrorString(e));
    return OMBO_ERR_CUDA;
  }
  OMBO_CHECK(device >= 0 && device < count, "ctx_create: device %d out of range (0..%d)", device, count - 1);
  OMBO_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  OMBO_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    ombo_set_error("ctx_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
                   prop.major, prop.minor);
    return OMBO_ERR_UNSUPPORTED;
  }
  {   // stream-ordered allocations (the likelihood workspace of concurrent fits) keep their blocks across calls
    cudaMemPool_t mp;
    unsigned long long keep = ~0ull;
    OMBO_CUDA(cudaDeviceGetDefaultMemPool(&mp, device));
    OMBO_CUDA(cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep));
  }
  ombo_ctx *c = new ombo_ctx();
  memset(c, 0, sizeof(*c));
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  {   // environment knobs: read here, once, never on the launch path
    auto geti = [](const char *name, int dflt) { const char *e = getenv(name); return e ? atoi(e) : dflt; };
    ombo_knobs &k = c->knobs;
    k.fast_dbg = geti("OMBO_FAST_DBG", 0);
    k.fast_profile = geti("OMBO_FAST_PROFILE", 0);
    k.fast_gen_warps = geti("OMBO_FAST_GEN_WARPS", 0);
    k.f8_max_run = geti("OMBO_F8_MAXRUN", 0);
    { const char *e = getenv("OMBO_F8_TG"); k.f8_tg = e ? atof(e) : 3.0; }
    k.chunk_log2 = geti("OMBO_CHUNK_LOG2", OMBO_CHUNK_DEV_LOG2);
    if (k.chunk_log2 < 10) k.chunk_log2 = 10;
    if (k.chunk_log2 > 26) k.chunk_log2 = 26;
    k.no_f8c = getenv("OMBO_NO_F8C") != nullptr;
    { const char *e = getenv("OMBO_F8C_KAPPA"); k.f8c_kappa = e ? atof(e) : OMBO_F8C_KAPPA_DEFAULT; }
    k.acq_fp64 = getenv("OMBO_ACQ_FP64") != nullptr;
    k.no_fuse = getenv("OMBO_NO_FUSE") != nullptr;
    k.no_prune = getenv("OMBO_NO_PRUNE") != nullptr;
    k.prune_depth = geti("OMBO_PRUNE_DEPTH", 1) >= 2 ? 2 : 1;
    { const char *e = getenv("OMBO_PRUNE_CAP"); k.prune_cap = e ? atoll(e) : 0; }
    k.prune_log = getenv("OMBO_PRUNE_LOG") != nullptr;
    k.prune_stage1 = geti("OMBO_PRUNE_STAGE1", 1) != 0;
    { const char *e = getenv("OMBO_PRUNE_STAGE1_CAP"); k.prune_cap1 = e ? atoll(e) : 0; }
    { const char *e = getenv("OMBO_STAGE1_KERNEL"); k.stage1_mean8 = e && strcmp(e, "mean8") == 0; }
  }
  OMBO_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    OMBO_CUDA(cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
    OMBO_CUDA(cudaEventCreateWithFlags(&c->ev_consumed[i], cudaEventDisableTiming));
  }
  OMBO_CUDA(cudaMalloc(&c->ws_best, 64));
  OMBO_CUDA(cudaMallocHost((void **)&c->pinned_best, 64));
  *out = c;
  return OMBO_OK;
}

int ombo_ctx_destroy(ombo_ctx *c) {
  if (!c) return OMBO_OK;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  if (c->ws_post) cudaFree(c->ws_post);
  if (c->ws_scratch) cudaFree(c->ws_scratch);
  if (c->ws_partial) cudaFree(c->ws_partial);
  if (c->ws_box) cudaFree(c->ws_box);
  for (int i = 0; i < 2; ++i) {
    if (c->ws_stage[i]) cudaFree(c->ws_stage[i]);
    cudaEventDestroy(c->ev_copied[i]);
    cudaEventDestroy(c->ev_consumed[i]);
  }
  if (c->prof_ev[0]) for (int i = 0; i < 2 * OMBO_PROF_MAX; ++i) cudaEventDestroy(c->prof_ev[i]);
  if (c->prof_dev) cudaFree(c->prof_dev);
  for (int i = 0; i < 2; ++i) if (c->f8_sched[i]) cudaFree(c->f8_sched[i]);
  if (c->ws_prune) cudaFree(c->ws_prune);
  if (c->ws_prune1) cudaFree(c->ws_prune1);
  if (c->ws_topk) cudaFree(c->ws_topk);
  if (c->ws_boxprep) cudaFree(c->ws_boxprep);
  if (c->ws_best) cudaFree(c->ws_best);
  if (c->pinned_best) cudaFreeHost(c->pinned_best);
  cudaStreamDestroy(c->copy_stream);
  delete c;
  return OMBO_OK;
}

int ombo_n_pad(int n) { return gp_layout(n, 1).n_pad; }

int ombo_gp_state_bytes(int n, int d, size_t *bytes) {
  OMBO_CHECK(n >= 1 && n <= OMBO_MAX_TRAIN, "gp_state_bytes: n=%d out of range (1..%d)", n, OMBO_MAX_TRAIN);
  OMBO_CHECK(d >= 1 && d <= OMBO_MAX_DIM, "gp_state_bytes: d=%d out of range (1..%d)", d, OMBO_MAX_DIM);
  OMBO_CHECK(bytes != nullptr, "gp_state_bytes: bytes is NULL");
  *bytes = gp_layout(n, d).bytes;
  return OMBO_OK;
}

int ombo_gp_state_field(int n, int d, int field, size_t *off, size_t *count) {
  OMBO_CHECK(n >= 1 && n <= OMBO_MAX_TRAIN && d >= 1 && d <= OMBO_MAX_DIM, "gp_state_field: bad n/d");
  OMBO_CHECK(off && count, "gp_state_field: NULL output");
  GpLayout L = gp_layout(n, d);
  size_t np = L.n_pad;
  switch (field) {
    case OMBO_FIELD_L: *off = L.off_L; *count = np * np; break;
    case OMBO_FIELD_LINV: *off = L.off_Linv; *count = np * np; break;
    case OMBO_FIELD_ALPHA: *off = L.off_alpha; *count = np; break;
    case OMBO_FIELD_XS: *off = L.off_xs; *count = (size_t)d * np; break;
    case OMBO_FIELD_STATUS: *off = L.off_status; *count = 4; break;
    case OMBO_FIELD_BHI: *off = L.off_bhi; *count = np * np; break;
    case OMBO_FIELD_BLO: *off = L.off_blo; *count = np * np; break;
    case OMBO_FIELD_XS32: *off = L.off_xs32; *count = np * 32; break;
    case OMBO_FIELD_ALPHA32: *off = L.off_alpha32; *count = np; break;
    default: ombo_set_error("gp_state_field: unknown field %d", field); return OMBO_ERR_INVALID;
  }
  return OMBO_OK;
}

int ombo_gp_refresh(ombo_ctx *ctx, const ombo_gp_spec *sp, void *state, void *stream) {
  OMBO_CHECK(ctx && sp && state, "gp_refresh: NULL argument");
  OMBO_CHECK(sp->n >= 1 && sp->n <= OMBO_MAX_TRAIN, "gp_refresh: n=%d out of range", sp->n);
  OMBO_CHECK(sp->d >= 1 && sp->d <= OMBO_MAX_DIM, "gp_refresh: d=%d out of range", sp->d);
  OMBO_CHECK(sp->kernel == OMBO_KERNEL_MATERN52 || sp->kernel == OMBO_KERNEL_RBF, "gp_refresh: unknown kernel %d", sp->kernel);
  OMBO_CHECK(sp->X && sp->y && sp->ell, "gp_refresh: NULL X/y/ell");
  OMBO_CHECK(sp->sigma_f2 > 0.0 && sp->sigma_n2 >= 0.0 && sp->jitter >= 0.0, "gp_refresh: bad hyper-parameters");
  for (int j = 0; j < sp->d; ++j) OMBO_CHECK(sp->ell[j] > 0.0, "gp_refresh: ell[%d] <= 0", j);
  OMBO_CUDA(cudaSetDevice(ctx->device));
  return ombo_refresh_impl(ctx, sp, state, (cudaStream_t)stream);
}

int ombo_gp_nlml_grad(ombo_ctx *ctx, const ombo_gp_spec *sp, void *state, double *out_host, void *stream) {
  OMBO_CHECK(ctx && sp && state && out_host, "gp_nlml_grad: NULL argument");
  OMBO_CHECK(sp->n >= 1 && sp->n <= OMBO_MAX_TRAIN && sp->d >= 1 && sp->d <= OMBO_MAX_DIM, "gp_nlml_grad: n/d out of range");
  OMBO_CHECK(sp->kernel == OMBO_KERNEL_MATERN52 || sp->kernel == OMBO_KERNEL_RBF, "gp_nlml_grad: unknown kernel");
  OMBO_CHECK(sp->X && sp->y && sp->ell, "gp_nlml_grad: NULL X/y/ell");
  OMBO_CHECK(sp->sigma_f2 > 0.0 && sp->sigma_n2 >= 0.0 && sp->jitter >= 0.0, "gp_nlml_grad: bad hyper-parameters");
  for (int j = 0; j < sp->d; ++j) OMBO_CHECK(sp->ell[j] > 0.0, "gp_nlml_grad: ell[%d] <= 0", j);
  OMBO_CUDA(cudaSetDevice(ctx->device));
  return ombo_nlml_grad_impl(ctx, sp, state, out_host, (cudaStream_t)stream);
}

}  // extern "C"

int ombo_validate_score(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const ombo_acq *acq,
                        int precision) {
  OMBO_CHECK(ctx && gps && pool && acq, "score: NULL argument");
  OMBO_CHECK(n_gp >= 1 && n_gp <= OMBO_MAX_GP, "score: n_gp=%d out of range (1..%d)", n_gp, OMBO_MAX_GP);
  OMBO_CHECK(precision == OMBO_PREC_FP64 || precision == OMBO_PREC_FAST, "score: unknown precision %d", precision);
  OMBO_CHECK(pool->m >= 0, "score: negative m");
  OMBO_CHECK(pool->d >= 1 && pool->d <= OMBO_MAX_DIM, "score: d=%d out of range", pool->d);
  OMBO_CHECK(pool->dtype == 0 || pool->dtype == 1, "score: pool dtype must be 0 (f64) or 1 (f32)");
  for (int g = 0; g < n_gp; ++g) {
    OMBO_CHECK(gps[g].state != nullptr, "score: gp %d has no state", g);
    OMBO_CHECK(gps[g].d == pool->d, "score: gp %d has d=%d but the pool has d=%d", g, gps[g].d, pool->d);
    OMBO_CHECK(gps[g].n >= 1 && gps[g].n <= OMBO_MAX_TRAIN, "score: gp %d: n out of range", g);
  }
  const int k = acq->n_obj;
  switch (acq->kind) {
    case OMBO_ACQ_NONE: break;
    case OMBO_ACQ_EHVI2D:
      OMBO_CHECK(n_gp >= 2 && acq->stripes && acq->n_pf >= 1, "EHVI2D needs 2 GPs and the PF stripes");
      break;
    case OMBO_ACQ_EHVI3D:
      OMBO_CHECK(k >= 2 && k <= OMBO_MAX_OBJ && n_gp >= k && acq->cache && acq->n_samples >= 1, "EHVI3D needs n_obj GPs and the sample cache");
      break;
    case OMBO_ACQ_EXPECTED_DECOMP:
      OMBO_CHECK(k >= 1 && k <= OMBO_MAX_OBJ && n_gp >= k && acq->cache && acq->n_samples >= 1, "EXPECTED_DECOMP needs n_obj GPs and the sample cache");
      OMBO_CHECK(acq->scalarisation >= 0 && acq->scalarisation <= OMBO_SC_APD, "unknown scalarisation %d", acq->scalarisation);
      break;
    case OMBO_ACQ_EI: break;
    case OMBO_ACQ_CONSTRAINED_EI: break;
    case OMBO_ACQ_PARETO_EI: OMBO_CHECK(n_gp >= 2, "PARETO_EI needs 2 GPs"); break;
    case OMBO_ACQ_HV_POI:
      OMBO_CHECK(n_gp >= 2 && acq->n_obj == 2 && acq->cells && acq->n_cells >= 1, "HV_POI needs 2 GPs, n_obj = 2 and the cells");
      break;
    case OMBO_ACQ_EHVI_BOX:
    case OMBO_ACQ_EHVI_BOX_FEAS:
    case OMBO_ACQ_HV_POI_BOX:
      OMBO_CHECK(k >= 2 && k <= OMBO_MAX_OBJ && n_gp >= k && acq->stripes && acq->cells,
                 "EHVI_BOX needs 2 <= n_obj <= %d, n_obj GPs, the breakpoint table and the boxes", OMBO_MAX_OBJ);
      OMBO_CHECK(acq->kind != OMBO_ACQ_EHVI_BOX_FEAS || n_gp >= k + 1,
                 "EHVI_BOX_FEAS needs n_obj objective GPs and at least one constraint GP (n_gp = %d, n_obj = %d)",
                 n_gp, k);
      OMBO_CHECK(acq->n_pf >= 2 && acq->n_pf <= OMBO_EHVI_BOX_MAX_BREAKS,
                 "EHVI_BOX: %d breakpoints per objective, supported 2..%d (a front of up to %d points)", acq->n_pf,
                 OMBO_EHVI_BOX_MAX_BREAKS, OMBO_EHVI_BOX_MAX_BREAKS - 2);
      OMBO_CHECK(acq->n_cells >= 1 && acq->n_cells <= OMBO_EHVI_BOX_MAX_BOXES,
                 "EHVI_BOX: %d boxes, supported 1..%d", acq->n_cells, OMBO_EHVI_BOX_MAX_BOXES);
      break;
    default: ombo_set_error("score: unknown acquisition kind %d", acq->kind); return OMBO_ERR_INVALID;
  }
  OMBO_CHECK(acq->semantics == OMBO_SEM_REFERENCE || acq->semantics == OMBO_SEM_EXACT, "score: unknown semantics");
  return OMBO_OK;
}

static void fill_pool_dev(PoolDev &pd, const ombo_pool *pool) {
  pd.X = nullptr; pd.dtype = pool->dtype; pd.d = pool->d; pd.index_base = pool->index_base; pd.seed = pool->seed;
  for (int j = 0; j < OMBO_MAX_DIM; ++j) {
    pd.lo[j] = (j < pool->d) ? pool->lo[j] : 0.0;
    pd.span[j] = (j < pool->d) ? pool->hi[j] - pool->lo[j] : 0.0;
  }
}

int ombo_score_pass(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const void *X_dev,
                    long long first, long long count, const ombo_acq *acq, int precision, double *out_mu,
                    double *out_var, double *out_acq, long long out_ld, ombo_best *best_dev, cudaStream_t s,
                    int bound_chunks) {
  PoolDev pd;
  fill_pool_dev(pd, pool);
  pd.X = X_dev;
  pd.index_base = pool->index_base + first;
  double *mu = out_mu ? out_mu + first : nullptr, *var = out_var ? out_var + first : nullptr;
  long long ld = out_ld;
  if (!mu || !var) {
    size_t want = (size_t)2 * n_gp * count * 8;
    int rc = ombo_ws_reserve(&ctx->ws_post, &ctx->ws_post_bytes, want);
    if (rc) return rc;
    mu = (double *)ctx->ws_post;
    var = mu + (size_t)n_gp * count;
    ld = count;
  }
  int fused = 0;
  // K4 + K5 fused behind the last K2 launch of the pass (fast mode, 2-D EHVI, nobody asked for the posterior itself):
  // the f8c kernel's epilogue warps evaluate the EHVI from registers and keep a per-CTA arg-max, so that model's
  // mu / var are never written and k_acquire does not run (ehvi2d_value is the same function either way).  The
  // launch that carries the acquisition must be a variance launch: model 1 in exact semantics, model 0 in reference
  // semantics (which reads only model 0's variance, so model 1 goes first through the mean-only kernel).
  const bool fuse_candidate = precision == OMBO_PREC_FAST && n_gp == 2 && acq->kind == OMBO_ACQ_EHVI2D && !out_mu &&
                              !out_var && !ctx->knobs.no_fuse && !ctx->knobs.acq_fp64 && (out_acq || best_dev);
  const int fuse_g = fuse_candidate ? (acq->semantics == OMBO_SEM_EXACT ? 1 : 0) : -1;
  for (int step = 0; step < n_gp; ++step) {
    const int g = fuse_g == 0 ? n_gp - 1 - step : step;          // the fused model's launch comes last
    GpDev gd = gp_dev_view(gps[g]);
    // K2 is skipped for GPs whose variance nothing reads (the caller did not ask for the posterior and
    // the acquisition ignores it): reference-semantics EHVI / EHVI_3D / expected decomposition scale
    // every objective by model 0's variance (util_functions.py:233), KEEP reads only the Pareto
    // model's mean (keep.py:149)
    bool want_var = true;
    if (!out_var) {
      const bool ref = acq->semantics == OMBO_SEM_REFERENCE;
      switch (acq->kind) {
        case OMBO_ACQ_EHVI2D: case OMBO_ACQ_EHVI3D: case OMBO_ACQ_EXPECTED_DECOMP:
          want_var = ref ? (g == 0) : (g < (acq->kind == OMBO_ACQ_EHVI2D ? 2 : acq->n_obj)); break;
        case OMBO_ACQ_EI: want_var = (g == 0); break;
        case OMBO_ACQ_PARETO_EI: want_var = (g == 1); break;
        case OMBO_ACQ_HV_POI: want_var = (g < 2); break;
        case OMBO_ACQ_EHVI_BOX: case OMBO_ACQ_HV_POI_BOX: want_var = (g < acq->n_obj); break;
        default: want_var = true;           // EHVI_BOX_FEAS: the objectives and every constraint
      }
    }
    FuseAcq fq;
    const bool try_fuse = g == fuse_g && step == n_gp - 1 && want_var;
    if (try_fuse) {
      const int o = 1 - g;
      memset(&fq, 0, sizeof(fq));
      fq.n_pf = acq->n_pf; fq.exact = acq->semantics == OMBO_SEM_EXACT;
      fq.c00 = (float)acq->cache_c00; fq.c01 = (float)acq->cache_c01;
      fq.self_model = g;
      fq.mu_other = mu + (size_t)o * ld;
      fq.var_other = fq.exact ? var + (size_t)o * ld : nullptr;      // reference semantics never reads model 1's variance
      fq.stripes = acq->stripes;
      fq.out_acq = out_acq ? out_acq + first : nullptr;
      fq.index_base = pd.index_base;
    }
    int rc = (precision == OMBO_PREC_FP64)
                 ? ombo_posterior_fp64(ctx, gd, pd, count, mu + (size_t)g * ld, var + (size_t)g * ld, want_var, s)
                 : ombo_posterior_fast(ctx, gd, pd, count, mu + (size_t)g * ld, var + (size_t)g * ld, want_var, s,
                                       try_fuse ? &fq : nullptr, &fused, bound_chunks);
    if (rc) return rc;
  }
  if (fused) return best_dev ? ombo_argmax_merge(ctx, fused, best_dev, s) : OMBO_OK;
  if (acq->kind != OMBO_ACQ_NONE)
    return ombo_acquire(ctx, acq, n_gp, mu, var, count, ld, pd.index_base, out_acq ? out_acq + first : nullptr,
                        best_dev, s, precision == OMBO_PREC_FAST);
  return OMBO_OK;
}

// every pass of a pool (2^chunk_log2 candidates each) through score_pass
static int score_passes(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const ombo_acq *acq,
                        int precision, double *out_mu, double *out_var, double *out_acq, ombo_best *best_dev,
                        cudaStream_t s, int bound_chunks = 0) {
  const size_t esz = pool->dtype == 0 ? 8 : 4;
  const long long chunk = 1LL << ctx->knobs.chunk_log2;
  for (long long first = 0; first < pool->m; first += chunk) {
    long long count = pool->m - first < chunk ? pool->m - first : chunk;
    const void *X = pool->X ? (const char *)pool->X + (size_t)first * pool->d * esz : nullptr;
    int rc = ombo_score_pass(ctx, gps, n_gp, pool, X, first, count, acq, precision, out_mu, out_var, out_acq, pool->m,
                        best_dev, s, bound_chunks);
    if (rc) return rc;
  }
  return OMBO_OK;
}

// ---- pruned arg-max (fast mode, exact-semantics 2-D EHVI, only `best` asked for) ---------------------------------
// The bound pass scores every candidate with its exact mean and an upper bound on each variance (posterior_fast8.cu,
// BOUND schedule: the first OMBO_PRUNE_DEPTH chunks of V).  Over a valid front the exact EHVI never decreases in
// either sigma (DESIGN.md section 4), so that score UB_i bounds the candidate's value from above.  The candidate with
// the largest UB is scored in full; its value v0 is a lower bound on the pool's best, and only candidates with
// UB_i >= v0 - tau can reach it.  Those are gathered into an explicit pool and scored in full, through the same
// fused path as the unpruned call, so the winner and its value are the unpruned call's.
//
// tau covers the FP32 evaluation of ehvi2d_value on both sides (the computed function is monotone in sigma only up
// to rounding): twice the FP32 contract of the acquisition (relative 1e-3 of the value, DESIGN.md section 4).
#define OMBO_PRUNE_TAU 2e-3

struct PruneHdr {                 // device, read back by one copy after the selection
  ombo_best ub;                   // largest upper bound (value, global index)
  ombo_best v0;                   // full score of that candidate (index: 0, it was scored alone)
  ombo_best loc;                  // best survivor (index: position in the survivor list)
  long long n_sel;                // survivors
};
static_assert(sizeof(PruneHdr) <= 64, "PruneHdr is read back through the context's 64-byte pinned buffer");

struct PruneKeep {                // survivor test of local candidate i
  const double *ub;
  const PruneHdr *h;
  __device__ bool operator()(long long i) const {
    const double u = ub[i];
    return isnan(u) || u >= h->v0.value - OMBO_PRUNE_TAU * h->ub.value;
  }
};

__global__ void k_prune_init(PruneHdr *h) {
  h->ub.value = h->v0.value = h->loc.value = -INFINITY;
  h->ub.index = h->v0.index = h->loc.index = -1;
  h->n_sel = 0;
}

// rows of the listed local candidates (idx == NULL: the one with the largest bound) into an explicit pool, converted
// exactly as the kernels read them: the f32 values of an f32 pool, the f64 coordinates of an f64 or counter pool
__global__ void k_prune_gather(PoolDev pool, long long m, const long long *__restrict__ idx,
                               const PruneHdr *__restrict__ h, long long n, void *__restrict__ out, int out_f32) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n * pool.d) return;
  const long long r = e / pool.d;
  const int j = (int)(e % pool.d);
  long long c = idx ? idx[r] : h->ub.index - pool.index_base;
  if (c < 0 || c >= m) c = 0;                     // no finite bound: the host falls back before using this row
  const double x = ombo_pool_coord(pool, c, j);
  if (out_f32) ((float *)out)[e] = (float)x;
  else ((double *)out)[e] = x;
}

// the threshold candidate and the best survivor, mapped to global indices, merged into the running best
__global__ void k_prune_merge(const PruneHdr *__restrict__ h, const long long *__restrict__ idx, long long base,
                              ombo_best *__restrict__ best) {
  BestPair b;
  b.v = h->v0.value; b.i = h->ub.index;
  if (h->loc.index >= 0) {
    const long long gi = base + idx[h->loc.index];
    if (better(h->loc.value, gi, b.v, b.i)) { b.v = h->loc.value; b.i = gi; }
  }
  if (best->index < 0 || better(b.v, b.i, best->value, best->index)) { best->value = b.v; best->index = b.i; }
}

static bool prune_eligible(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const ombo_acq *acq,
                           int precision, const double *out_mu, const double *out_acq, const ombo_best *best_dev,
                           cudaStream_t s) {
  if (precision != OMBO_PREC_FAST || n_gp != 2 || acq->kind != OMBO_ACQ_EHVI2D || acq->semantics != OMBO_SEM_EXACT ||
      !(acq->reserved & OMBO_ACQ_FRONT_VALID) || out_mu || out_acq || !best_dev || pool->m < 1 ||
      ctx->knobs.no_prune || ctx->knobs.no_fuse || ctx->knobs.acq_fp64)
    return false;
  // timing experiments (OMBO_FAST_DBG) compute garbage; the bound is derived from the pass schedule, so a full launch
  // on the rolling schedule (OMBO_F8_MAXRUN) would not share chunk 0's accumulation order with it
  if (ctx->knobs.fast_dbg || ctx->knobs.f8_max_run > 0) return false;
  for (int g = 0; g < 2; ++g)
    if (!(gps[g].reserved & OMBO_GP_F8C_PLANES)) return false;
  // model 1's launch must carry the fused acquisition in the bound pass and in the full one
  const GpDev g1 = gp_dev_view(gps[1]);
  return ombo_f8_can_fuse(ctx, g1, acq->n_pf, ctx->knobs.prune_depth, s) && ombo_f8_can_fuse(ctx, g1, acq->n_pf, 0, s);
}

// the depth-1 path: the BOUND pass over the pool, its threshold and survivors; *done = false: nothing was merged
// into best_dev and the caller scores the pool in full
static int prune_depth1(ombo_ctx *ctx, const ombo_gp *gps, const ombo_pool *pool, const ombo_acq *acq,
                        ombo_best *best_dev, cudaStream_t s, bool *done) {
  *done = false;
  const long long m = pool->m;
  const long long cap = ctx->knobs.prune_cap > 0 ? ctx->knobs.prune_cap : std::max(1LL << 16, m / 64);
  const int out_f32 = pool->X && pool->dtype == 1;
  const size_t resz = out_f32 ? 4 : 8;
  auto up = [](size_t b) { return (b + 255) / 256 * 256; };
  const cub::CountingInputIterator<long long> ids(0);
  size_t cub_bytes = 0;
  OMBO_CUDA(cub::DeviceSelect::If(nullptr, cub_bytes, ids, (long long *)nullptr, (long long *)nullptr, m,
                                  PruneKeep{nullptr, nullptr}, s));
  const size_t o_ub = up(sizeof(PruneHdr)), o_sel = o_ub + up((size_t)m * 8), o_rows = o_sel + up((size_t)m * 8),
               o_cub = o_rows + up((size_t)std::min(cap, m) * pool->d * resz);
  // O(m) workspace: a pool too large for it is scored the unpruned way, in its bounded passes
  if (ombo_ws_reserve(&ctx->ws_prune, &ctx->ws_prune_bytes, o_cub + cub_bytes)) {
    (void)cudaGetLastError();                       // the failed allocation is not sticky; clear it
    return OMBO_OK;
  }
  int rc;
  char *ws = (char *)ctx->ws_prune;
  PruneHdr *h = (PruneHdr *)ws;
  double *ub = (double *)(ws + o_ub);
  long long *sel = (long long *)(ws + o_sel);
  void *rows = ws + o_rows;
  k_prune_init<<<1, 1, 0, s>>>(h);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  // bound pass: UB of every candidate and the largest
  rc = score_passes(ctx, gps, 2, pool, acq, OMBO_PREC_FAST, nullptr, nullptr, ub, &h->ub, s, ctx->knobs.prune_depth);
  if (rc) return rc;
  // threshold: the full score of the candidate with the largest bound
  PoolDev pd;
  fill_pool_dev(pd, pool);
  pd.X = pool->X;
  k_prune_gather<<<1, 32, 0, s>>>(pd, m, nullptr, h, 1, rows, out_f32);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  ombo_pool sub = *pool;
  sub.X = rows; sub.dtype = out_f32; sub.m = 1; sub.index_base = 0;
  rc = score_passes(ctx, gps, 2, &sub, acq, OMBO_PREC_FAST, nullptr, nullptr, nullptr, &h->v0, s);
  if (rc) return rc;
  // survivors, in ascending index order
  OMBO_CUDA(cub::DeviceSelect::If(ws + o_cub, cub_bytes, ids, sel, &h->n_sel, m, PruneKeep{ub, h}, s));
  ctx->launches += 1;
  PruneHdr hh;
  OMBO_CUDA(cudaMemcpyAsync(ctx->pinned_best, h, sizeof(PruneHdr), cudaMemcpyDeviceToHost, s));
  OMBO_CUDA(cudaStreamSynchronize(s));
  memcpy(&hh, ctx->pinned_best, sizeof(PruneHdr));
  if (ctx->knobs.prune_log)
    fprintf(stderr, "[prune] m %lld survivors %lld ub_max %.9g at %lld v0 %.9g cap %lld\n", m, hh.n_sel, hh.ub.value,
            (long long)hh.ub.index, hh.v0.value, cap);
  // a threshold at or below zero prunes nothing worth the second pass; too many survivors cost more than they save
  if (!std::isfinite(hh.ub.value) || !(hh.v0.value - OMBO_PRUNE_TAU * hh.ub.value > 0.0) || hh.n_sel > cap)
    return OMBO_OK;
  if (hh.n_sel > 0) {
    const long long n = hh.n_sel;
    k_prune_gather<<<(unsigned)((n * pool->d + 255) / 256), 256, 0, s>>>(pd, m, sel, h, n, rows, out_f32);
    ctx->launches += 1;
    OMBO_CUDA(cudaGetLastError());
    sub.m = n;
    rc = score_passes(ctx, gps, 2, &sub, acq, OMBO_PREC_FAST, nullptr, nullptr, nullptr, &h->loc, s);
    if (rc) return rc;
  }
  k_prune_merge<<<1, 1, 0, s>>>(h, sel, pool->index_base, best_dev);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  *done = true;
  return OMBO_OK;
}

// ---- stage 1 of the pruned arg-max: the mean-only bound (posterior_mean8.cu) ---------------------------------------
// UB1 (both means exact, each variance replaced by its prior bound) is computed for every candidate in one launch.
// The threshold v0 is the largest full score among the per-CTA maxima of UB1 (one candidate per CTA of the launch,
// the global maximum among them); candidates with UB1 >= v0 - tau UB1_max (or NaN) survive, by the argument above
// with UB1 in place of UB.  The survivors are gathered into an explicit pool and go through the depth-1 path
// unchanged; a gathered subset reproduces mu, var and the values bit for bit, so the winner and its value are the
// unpruned call's.  Too many survivors (or no positive threshold): the depth-1 path takes the whole pool.

// rows of the per-CTA maxima (partials of the stage-1 launch) into an explicit pool, and their local indices
__global__ void k_prune1_top(PoolDev pool, long long m, const ombo_best *__restrict__ partials, int n,
                             long long *__restrict__ top_idx, void *__restrict__ out, int out_f32) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n * pool.d) return;
  const int r = e / pool.d, j = e % pool.d;
  long long c = partials[r].index - pool.index_base;
  if (c < 0 || c >= m) c = 0;                     // a CTA without candidates: row 0 stands in (a real candidate)
  if (j == 0) top_idx[r] = c;
  const double x = ombo_pool_coord(pool, c, j);
  if (out_f32) ((float *)out)[e] = (float)x;
  else ((double *)out)[e] = x;
}

// the best threshold candidate and the best survivor of stage 2, mapped to global indices, into the running best
__global__ void k_prune1_merge(const PruneHdr *__restrict__ h, const long long *__restrict__ top_idx,
                               const long long *__restrict__ sel, long long base, ombo_best *__restrict__ best) {
  BestPair b;
  b.v = -INFINITY; b.i = -1;
  if (h->v0.index >= 0) { b.v = h->v0.value; b.i = base + top_idx[h->v0.index]; }
  if (h->loc.index >= 0) {
    const long long gi = base + sel[h->loc.index];
    if (b.i < 0 || better(h->loc.value, gi, b.v, b.i)) { b.v = h->loc.value; b.i = gi; }
  }
  if (b.i >= 0 && (best->index < 0 || better(b.v, b.i, best->value, best->index))) {
    best->value = b.v; best->index = b.i;
  }
}

static int score_pruned(ombo_ctx *ctx, const ombo_gp *gps, const ombo_pool *pool, const ombo_acq *acq,
                        ombo_best *best_dev, cudaStream_t s, bool *done) {
  *done = false;
  const GpDev gd[2] = {gp_dev_view(gps[0]), gp_dev_view(gps[1])};
  // stage 1 on the tensor core where it covers the shape and its margin stays small for this pool (decided below),
  // else (or with OMBO_STAGE1_KERNEL=mean8) the exact-mean kernel
  bool tc = !ctx->knobs.stage1_mean8 && ombo_stage1_tc_covers(gd, acq->n_pf);
  if (!ctx->knobs.prune_stage1 || !(tc || ombo_mean8_covers(gd, acq->n_pf)))
    return prune_depth1(ctx, gps, pool, acq, best_dev, s, done);
  const long long m = pool->m;
  const long long cap = ctx->knobs.prune_cap1 > 0 ? ctx->knobs.prune_cap1 : std::max(1LL << 16, m / 8);
  const int n_top = ctx->num_sms;                 // the most CTAs stage 1 launches: one threshold row each
  const int out_f32 = pool->X && pool->dtype == 1;
  const size_t resz = out_f32 ? 4 : 8;
  auto up = [](size_t b) { return (b + 255) / 256 * 256; };
  const cub::CountingInputIterator<long long> ids(0);
  size_t cub_bytes = 0;
  OMBO_CUDA(cub::DeviceSelect::If(nullptr, cub_bytes, ids, (long long *)nullptr, (long long *)nullptr, m,
                                  PruneKeep{nullptr, nullptr}, s));
  const size_t o_ext = up(sizeof(PruneHdr)), o_top = o_ext + 256, o_trows = o_top + up((size_t)n_top * 8),
               o_ub = o_trows + up((size_t)n_top * pool->d * resz), o_sel = o_ub + up((size_t)m * 8),
               o_rows = o_sel + up((size_t)m * 8), o_cub = o_rows + up((size_t)std::min(cap, m) * pool->d * resz);
  if (ombo_ws_reserve(&ctx->ws_prune1, &ctx->ws_prune1_bytes, o_cub + cub_bytes)) {
    (void)cudaGetLastError();
    return prune_depth1(ctx, gps, pool, acq, best_dev, s, done);
  }
  int rc;
  char *ws = (char *)ctx->ws_prune1;
  PruneHdr *h = (PruneHdr *)ws;
  long long *top_idx = (long long *)(ws + o_top);
  void *trows = ws + o_trows;
  double *ub = (double *)(ws + o_ub);
  long long *sel = (long long *)(ws + o_sel);
  void *rows = ws + o_rows;
  k_prune_init<<<1, 1, 0, s>>>(h);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  PoolDev pd;
  fill_pool_dev(pd, pool);
  pd.X = pool->X;
  if (tc) {
    rc = ombo_stage1_tc_useful(ctx, gd, pd, m, ws + o_ext, &tc, s);
    if (rc) return rc;
    if (!tc && !ombo_mean8_covers(gd, acq->n_pf)) return prune_depth1(ctx, gps, pool, acq, best_dev, s, done);
  }
  // stage 1: UB1 of every candidate, the per-CTA maxima (ctx->ws_partial) and the largest
  int n_cta = 0;
  rc = tc ? ombo_stage1_tc_bound(ctx, gd, pd, m, acq->stripes, acq->n_pf, (float)acq->cache_c00,
                                 (float)acq->cache_c01, ub, &h->ub, nullptr, nullptr, &n_cta, s)
          : ombo_mean8_bound(ctx, gd, pd, m, acq->stripes, acq->n_pf, (float)acq->cache_c00, (float)acq->cache_c01, ub,
                             &h->ub, nullptr, &n_cta, s);
  if (rc) return rc;
  k_prune1_top<<<(unsigned)((n_cta * pool->d + 255) / 256), 256, 0, s>>>(pd, m, (const ombo_best *)ctx->ws_partial,
                                                                         n_cta, top_idx, trows, out_f32);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  // threshold: the best full score among them (local index into top_idx)
  ombo_pool sub = *pool;
  sub.X = trows; sub.dtype = out_f32; sub.m = n_cta; sub.index_base = 0;
  rc = score_passes(ctx, gps, 2, &sub, acq, OMBO_PREC_FAST, nullptr, nullptr, nullptr, &h->v0, s);
  if (rc) return rc;
  OMBO_CUDA(cub::DeviceSelect::If(ws + o_cub, cub_bytes, ids, sel, &h->n_sel, m, PruneKeep{ub, h}, s));
  ctx->launches += 1;
  PruneHdr hh;
  OMBO_CUDA(cudaMemcpyAsync(ctx->pinned_best, h, sizeof(PruneHdr), cudaMemcpyDeviceToHost, s));
  OMBO_CUDA(cudaStreamSynchronize(s));
  memcpy(&hh, ctx->pinned_best, sizeof(PruneHdr));
  if (ctx->knobs.prune_log)
    fprintf(stderr, "[prune1] m %lld survivors %lld ub_max %.9g at %lld v0 %.9g top %d cap %lld stage1 %s\n", m,
            hh.n_sel, hh.ub.value, (long long)hh.ub.index, hh.v0.value, n_cta, cap, tc ? "tc" : "mean8");
  if (!std::isfinite(hh.ub.value) || !(hh.v0.value - OMBO_PRUNE_TAU * hh.ub.value > 0.0) || hh.n_sel > cap)
    return prune_depth1(ctx, gps, pool, acq, best_dev, s, done);
  // stage 2: the depth-1 path on the survivors (local indices into sel), in full if it declines
  if (hh.n_sel > 0) {
    const long long n = hh.n_sel;
    k_prune_gather<<<(unsigned)((n * pool->d + 255) / 256), 256, 0, s>>>(pd, m, sel, h, n, rows, out_f32);
    ctx->launches += 1;
    OMBO_CUDA(cudaGetLastError());
    sub.X = rows; sub.m = n;
    bool done2 = false;
    rc = prune_depth1(ctx, gps, &sub, acq, &h->loc, s, &done2);
    if (rc) return rc;
    if (!done2) {
      rc = score_passes(ctx, gps, 2, &sub, acq, OMBO_PREC_FAST, nullptr, nullptr, nullptr, &h->loc, s);
      if (rc) return rc;
    }
  }
  k_prune1_merge<<<1, 1, 0, s>>>(h, top_idx, sel, pool->index_base, best_dev);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  *done = true;
  return OMBO_OK;
}

extern "C" {

int ombo_score(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const ombo_acq *acq,
               int precision, double *out_mu, double *out_var, double *out_acq, ombo_best *best_dev,
               void *stream) {
  int rc = ombo_validate_score(ctx, gps, n_gp, pool, acq, precision);
  if (rc) return rc;
  OMBO_CHECK((out_mu == nullptr) == (out_var == nullptr), "score: out_mu and out_var must both be given or both NULL");
  OMBO_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (best_dev) { rc = ombo_best_init(ctx, best_dev, s); if (rc) return rc; }
  if (prune_eligible(ctx, gps, n_gp, pool, acq, precision, out_mu, out_acq, best_dev, s)) {
    bool done = false;
    rc = score_pruned(ctx, gps, pool, acq, best_dev, s, &done);
    if (rc || done) return rc;
  }
  return score_passes(ctx, gps, n_gp, pool, acq, precision, out_mu, out_var, out_acq, best_dev, s);
}

int ombo_score_host(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const ombo_acq *acq,
                    int precision, ombo_best *best_host, void *stream) {
  int rc = ombo_validate_score(ctx, gps, n_gp, pool, acq, precision);
  if (rc) return rc;
  OMBO_CHECK(best_host != nullptr, "score_host: best_host is NULL");
  OMBO_CHECK(acq->kind != OMBO_ACQ_NONE, "score_host: needs an acquisition");
  OMBO_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  ombo_best *best_dev = (ombo_best *)ctx->ws_best;
  rc = ombo_best_init(ctx, best_dev, s);
  if (rc) return rc;
  const size_t esz = pool->dtype == 0 ? 8 : 4;
  if (pool->X) {
    size_t stage = (size_t)OMBO_CHUNK * pool->d * esz;
    if (ctx->ws_stage_bytes < stage) {
      OMBO_CUDA(cudaDeviceSynchronize());
      for (int i = 0; i < 2; ++i) {
        if (ctx->ws_stage[i]) OMBO_CUDA(cudaFree(ctx->ws_stage[i]));
        OMBO_CUDA(cudaMalloc(&ctx->ws_stage[i], stage));
      }
      ctx->ws_stage_bytes = stage;
    }
    // the copy stream must not run ahead of work already queued on `s`
    OMBO_CUDA(cudaEventRecord(ctx->ev_consumed[0], s));
    OMBO_CUDA(cudaEventRecord(ctx->ev_consumed[1], s));
  }
  int it = 0;
  for (long long first = 0; first < pool->m; first += OMBO_CHUNK, ++it) {
    long long count = pool->m - first < OMBO_CHUNK ? pool->m - first : OMBO_CHUNK;
    const void *X = nullptr;
    if (pool->X) {
      int b = it & 1;
      OMBO_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_consumed[b], 0));
      OMBO_CUDA(cudaMemcpyAsync(ctx->ws_stage[b], (const char *)pool->X + (size_t)first * pool->d * esz,
                                (size_t)count * pool->d * esz, cudaMemcpyHostToDevice, ctx->copy_stream));
      OMBO_CUDA(cudaEventRecord(ctx->ev_copied[b], ctx->copy_stream));
      OMBO_CUDA(cudaStreamWaitEvent(s, ctx->ev_copied[b], 0));
      X = ctx->ws_stage[b];
    }
    rc = ombo_score_pass(ctx, gps, n_gp, pool, X, first, count, acq, precision, nullptr, nullptr, nullptr, 0, best_dev, s);
    if (rc) return rc;
    if (pool->X) OMBO_CUDA(cudaEventRecord(ctx->ev_consumed[it & 1], s));
  }
  OMBO_CUDA(cudaMemcpyAsync(ctx->pinned_best, best_dev, sizeof(ombo_best), cudaMemcpyDeviceToHost, s));
  OMBO_CUDA(cudaStreamSynchronize(s));
  *best_host = *ctx->pinned_best;
  return OMBO_OK;
}

int ombo_acquire_posterior(ombo_ctx *ctx, const ombo_acq *acq, int n_gp, const double *mu, const double *var,
                           int64_t m, int64_t ld, int64_t index_base, double *out_acq, ombo_best *best_dev,
                           void *stream) {
  OMBO_CHECK(ctx && acq && mu && var, "acquire_posterior: NULL argument");
  OMBO_CHECK(n_gp >= 1 && n_gp <= OMBO_MAX_GP && m >= 0 && ld >= m, "acquire_posterior: bad sizes");
  ombo_pool fake;
  memset(&fake, 0, sizeof(fake));
  fake.d = 1; fake.m = m;
  ombo_gp gp_ok[OMBO_MAX_GP];
  for (int g = 0; g < n_gp; ++g) { gp_ok[g].state = (const void *)mu; gp_ok[g].d = 1; gp_ok[g].n = 1; }
  int rc = ombo_validate_score(ctx, gp_ok, n_gp, &fake, acq, OMBO_PREC_FP64);
  if (rc) return rc;
  OMBO_CHECK(acq->kind != OMBO_ACQ_NONE, "acquire_posterior: needs an acquisition kind");
  OMBO_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (best_dev) { rc = ombo_best_init(ctx, best_dev, s); if (rc) return rc; }
  return ombo_acquire(ctx, acq, n_gp, mu, var, m, ld, index_base, out_acq, best_dev, s);
}

int ombo_scalarise(ombo_ctx *ctx, const ombo_acq *acq, const double *F, int64_t m, double *out, void *stream) {
  OMBO_CHECK(ctx && acq && F && out, "scalarise: NULL argument");
  OMBO_CHECK(acq->n_obj >= 1 && acq->n_obj <= OMBO_MAX_OBJ, "scalarise: n_obj=%d out of range (1..%d)", acq->n_obj, OMBO_MAX_OBJ);
  OMBO_CHECK(acq->scalarisation >= 0 && acq->scalarisation <= OMBO_SC_APD, "scalarise: unknown scalarisation %d", acq->scalarisation);
  OMBO_CHECK(m >= 0, "scalarise: negative m");
  OMBO_CUDA(cudaSetDevice(ctx->device));
  return ombo_scalarise_impl(ctx, acq, F, m, out, (cudaStream_t)stream);
}

__global__ void k_pool_rows(PoolDev pool, long long first, long long count, double *__restrict__ out) {
  long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= count * pool.d) return;
  long long c = e / pool.d;
  int j = (int)(e % pool.d);
  out[e] = ombo_pool_coord(pool, first + c, j);
}

int ombo_pool_rows(ombo_ctx *ctx, const ombo_pool *pool, int64_t index, int64_t count, double *out, void *stream) {
  OMBO_CHECK(ctx && pool && out, "pool_rows: NULL argument");
  OMBO_CHECK(pool->d >= 1 && pool->d <= OMBO_MAX_DIM, "pool_rows: d out of range");
  OMBO_CHECK(index >= pool->index_base && count >= 0, "pool_rows: bad range");
  if (count == 0) return OMBO_OK;
  OMBO_CUDA(cudaSetDevice(ctx->device));
  PoolDev pd;
  fill_pool_dev(pd, pool);
  pd.X = pool->X;
  long long total = count * pool->d;
  k_pool_rows<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(pd, index - pool->index_base, count, out);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  return OMBO_OK;
}

__global__ void k_pool_gather(PoolDev pool, const long long *__restrict__ idx, long long count,
                              double *__restrict__ out) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= count * pool.d) return;
  out[e] = ombo_pool_coord(pool, idx[e / pool.d] - pool.index_base, (int)(e % pool.d));
}

int ombo_pool_gather(ombo_ctx *ctx, const ombo_pool *pool, const int64_t *index_dev, int64_t count, double *out,
                     void *stream) {
  OMBO_CHECK(ctx && pool && out && (index_dev || count == 0), "pool_gather: NULL argument");
  OMBO_CHECK(pool->d >= 1 && pool->d <= OMBO_MAX_DIM, "pool_gather: d out of range");
  OMBO_CHECK(pool->dtype == 0 || pool->dtype == 1, "pool_gather: pool dtype must be 0 (f64) or 1 (f32)");
  OMBO_CHECK(count >= 0, "pool_gather: negative count");
  if (count == 0) return OMBO_OK;
  OMBO_CUDA(cudaSetDevice(ctx->device));
  PoolDev pd;
  fill_pool_dev(pd, pool);
  pd.X = pool->X;
  const long long total = count * pool->d;
  k_pool_gather<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(pd, (const long long *)index_dev,
                                                                                   count, out);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  return OMBO_OK;
}

int ombo_pack_key(ombo_ctx *ctx, const ombo_best *best_dev, int64_t *key_dev, void *stream) {
  OMBO_CHECK(ctx && best_dev && key_dev, "pack_key: NULL argument");
  OMBO_CUDA(cudaSetDevice(ctx->device));
  return ombo_pack_key_impl(ctx, best_dev, (long long *)key_dev, (cudaStream_t)stream);
}

int ombo_pareto_mask(ombo_ctx *ctx, const double *Y, int n, int k, unsigned char *mask, void *stream) {
  OMBO_CHECK(ctx && Y && mask, "pareto_mask: NULL argument");
  OMBO_CHECK(n >= 1 && k >= 1 && k <= 8, "pareto_mask: need n >= 1 and 1 <= k <= 8 (got n=%d k=%d)", n, k);
  OMBO_CUDA(cudaSetDevice(ctx->device));
  return ombo_pareto_mask_impl(ctx, Y, n, k, mask, (cudaStream_t)stream);
}

int ombo_hypervolume(ombo_ctx *ctx, const double *P, int p, int k, const double *ref, double *hv_out, void *stream) {
  OMBO_CHECK(ctx && ref && hv_out && (P || p == 0), "hypervolume: NULL argument");
  OMBO_CHECK(k == 2 || k == 3, "hypervolume: 2 or 3 objectives (got %d)", k);
  OMBO_CHECK(p >= 0 && p <= 16384, "hypervolume: 0 <= p <= 16384 (got %d)", p);
  OMBO_CUDA(cudaSetDevice(ctx->device));
  return ombo_hypervolume_impl(ctx, P, p, k, ref, hv_out, (cudaStream_t)stream);
}

int ombo_cells_2d(ombo_ctx *ctx, const double *PF, int p, const double *ideal, const double *maxp, double *cells,
                  void *stream) {
  OMBO_CHECK(ctx && PF && ideal && maxp && cells, "cells_2d: NULL argument");
  OMBO_CHECK(p >= 1 && p <= 16384, "cells_2d: 1 <= p <= 16384 (got %d)", p);
  OMBO_CUDA(cudaSetDevice(ctx->device));
  return ombo_cells_2d_impl(ctx, PF, p, ideal, maxp, cells, (cudaStream_t)stream);
}

int ombo_ehvi_boxes(ombo_ctx *ctx, const double *PF, int p, int k, const double *ref, double *table, double *boxes,
                    int64_t boxes_cap, int *B_out, int64_t *n_boxes_out, void *stream) {
  OMBO_CHECK(ctx && ref && table && B_out && n_boxes_out && (PF || p == 0) && (boxes || boxes_cap == 0),
             "ehvi_boxes: NULL argument");
  OMBO_CHECK(k >= 2 && k <= OMBO_MAX_OBJ, "ehvi_boxes: 2 to %d objectives (got %d)", OMBO_MAX_OBJ, k);
  OMBO_CHECK(p >= 0 && p <= 16384, "ehvi_boxes: 0 <= p <= 16384 (got %d)", p);
  OMBO_CHECK(boxes_cap >= 0, "ehvi_boxes: negative boxes_cap");
  for (int c = 0; c < k; ++c) OMBO_CHECK(isfinite(ref[c]), "ehvi_boxes: ref[%d] is not finite", c);
  OMBO_CUDA(cudaSetDevice(ctx->device));
  long long nb = 0;
  const int rc = ombo_ehvi_boxes_impl(ctx, PF, p, k, ref, table, boxes, boxes_cap, B_out, &nb, (cudaStream_t)stream);
  *n_boxes_out = nb;
  return rc;
}

int ombo_posterior_joint_samples(ombo_ctx *ctx, const ombo_gp *gp, const double *Xc, int m, const double *Z,
                                 int n_samples, double diag_add, double *out, void *stream) {
  OMBO_CHECK(ctx && gp && gp->state && Xc && Z && out, "joint_samples: NULL argument");
  OMBO_CHECK(m >= 1 && m <= 16384, "joint_samples: 1 <= m <= 16384 (got %d)", m);
  OMBO_CHECK(n_samples >= 1 && n_samples <= 4096, "joint_samples: 1 <= n_samples <= 4096 (got %d)", n_samples);
  OMBO_CHECK(gp->n >= 1 && gp->d >= 1 && gp->d <= OMBO_MAX_DIM, "joint_samples: bad GP shape n=%d d=%d", gp->n, gp->d);
  OMBO_CHECK(diag_add >= 0.0, "joint_samples: diag_add must be >= 0");
  OMBO_CUDA(cudaSetDevice(ctx->device));
  return ombo_joint_samples_impl(ctx, *gp, Xc, m, Z, n_samples, diag_add, out, (cudaStream_t)stream);
}

int ombo_profile_enable(ombo_ctx *ctx, int enable) {
  OMBO_CHECK(ctx != nullptr, "profile_enable: NULL ctx");
  OMBO_CUDA(cudaSetDevice(ctx->device));
  if (enable && !ctx->prof_ev[0])
    for (int i = 0; i < 2 * OMBO_PROF_MAX; ++i) OMBO_CUDA(cudaEventCreate(&ctx->prof_ev[i]));
  ctx->prof_enabled = enable ? 1 : 0;
  ctx->prof_count = 0;
  return OMBO_OK;
}

int ombo_profile_read(ombo_ctx *ctx, int64_t *n_launches, double *total_ms) {
  OMBO_CHECK(ctx && n_launches && total_ms, "profile_read: NULL argument");
  OMBO_CUDA(cudaSetDevice(ctx->device));
  double tot = 0.0;
  for (int i = 0; i < ctx->prof_count; ++i) {
    OMBO_CUDA(cudaEventSynchronize(ctx->prof_ev[2 * i + 1]));
    float ms = 0.f;
    OMBO_CUDA(cudaEventElapsedTime(&ms, ctx->prof_ev[2 * i], ctx->prof_ev[2 * i + 1]));
    tot += ms;
  }
  *n_launches = ctx->prof_count;
  *total_ms = tot;
  ctx->prof_count = 0;
  return OMBO_OK;
}

// test hook (not part of the public header): mu and var of one GP with f8c planes over rows [0, m) of a pool, from
// the BOUND launch (bound_chunks >= 1: var is the upper bound of the pruned arg-max) or the full one (0), with
// gen_warps generator warps (8 / 16; 0: the context's choice)
int ombo_debug_posterior_bound(ombo_ctx *ctx, const ombo_gp *gp, const ombo_pool *pool, int bound_chunks,
                               int gen_warps, double *mu, double *var, void *stream) {
  OMBO_CHECK(ctx && gp && gp->state && pool && mu && var, "debug_posterior_bound: NULL argument");
  OMBO_CHECK(gp->reserved & OMBO_GP_F8C_PLANES, "debug_posterior_bound: the GP has no f8c planes");
  OMBO_CHECK(gp->d == pool->d && pool->m >= 0, "debug_posterior_bound: bad pool");
  OMBO_CHECK(bound_chunks >= 0 && bound_chunks <= 2 && (gen_warps == 0 || gen_warps == 8 || gen_warps == 16),
             "debug_posterior_bound: bound_chunks 0..2, gen_warps 0 / 8 / 16");
  OMBO_CUDA(cudaSetDevice(ctx->device));
  PoolDev pd;
  fill_pool_dev(pd, pool);
  pd.X = pool->X;
  const int keep = ctx->knobs.fast_gen_warps;
  ctx->knobs.fast_gen_warps = gen_warps;
  const int rc = ombo_posterior_fast(ctx, gp_dev_view(*gp), pd, pool->m, mu, var, true, (cudaStream_t)stream, nullptr,
                                     nullptr, bound_chunks);
  ctx->knobs.fast_gen_warps = keep;
  return rc;
}

// the stage-1 launch of the pruned arg-max on its own: mu [2][m] (the FP32 means as doubles), ub [m], the largest
// bound into *best_dev
int ombo_debug_mean8(ombo_ctx *ctx, const ombo_gp *gps, const ombo_pool *pool, const ombo_acq *acq, double *mu,
                     double *ub, ombo_best *best_dev, void *stream) {
  OMBO_CHECK(ctx && gps && pool && acq && mu && ub && best_dev, "debug_mean8: NULL argument");
  OMBO_CHECK(acq->kind == OMBO_ACQ_EHVI2D && acq->stripes && acq->n_pf >= 1, "debug_mean8: needs an EHVI2D spec");
  for (int g = 0; g < 2; ++g)
    OMBO_CHECK(gps[g].state && (gps[g].reserved & OMBO_GP_F8C_PLANES) && gps[g].d == pool->d,
               "debug_mean8: gp %d has no f8c planes or the wrong d", g);
  OMBO_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  PoolDev pd;
  fill_pool_dev(pd, pool);
  pd.X = pool->X;
  const GpDev gd[2] = {gp_dev_view(gps[0]), gp_dev_view(gps[1])};
  int rc = ombo_best_init(ctx, best_dev, s);
  if (rc) return rc;
  return ombo_mean8_bound(ctx, gd, pd, pool->m, acq->stripes, acq->n_pf, (float)acq->cache_c00,
                          (float)acq->cache_c01, ub, best_dev, mu, nullptr, s);
}

// the tensor-core stage-1 launch on its own: mu [2][m] (the stage-1 means), marg [2][m] (their margins M), ub [m],
// the largest bound into *best_dev; OMBO_ERR_UNSUPPORTED where the kernel does not cover the shape
int ombo_debug_stage1_tc(ombo_ctx *ctx, const ombo_gp *gps, const ombo_pool *pool, const ombo_acq *acq, double *mu,
                         double *marg, double *ub, ombo_best *best_dev, void *stream) {
  OMBO_CHECK(ctx && gps && pool && acq && mu && marg && ub && best_dev, "debug_stage1_tc: NULL argument");
  OMBO_CHECK(acq->kind == OMBO_ACQ_EHVI2D && acq->stripes && acq->n_pf >= 1, "debug_stage1_tc: needs an EHVI2D spec");
  for (int g = 0; g < 2; ++g)
    OMBO_CHECK(gps[g].state && (gps[g].reserved & OMBO_GP_F8C_PLANES) && gps[g].d == pool->d,
               "debug_stage1_tc: gp %d has no f8c planes or the wrong d", g);
  OMBO_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  PoolDev pd;
  fill_pool_dev(pd, pool);
  pd.X = pool->X;
  const GpDev gd[2] = {gp_dev_view(gps[0]), gp_dev_view(gps[1])};
  int rc = ombo_best_init(ctx, best_dev, s);
  if (rc) return rc;
  return ombo_stage1_tc_bound(ctx, gd, pd, pool->m, acq->stripes, acq->n_pf, (float)acq->cache_c00,
                              (float)acq->cache_c01, ub, best_dev, mu, marg, nullptr, s);
}

int64_t ombo_launch_count(ombo_ctx *ctx, int reset) {
  if (!ctx) return 0;
  int64_t v = ctx->launches;
  if (reset) ctx->launches = 0;
  return v;
}

}  // extern "C"
