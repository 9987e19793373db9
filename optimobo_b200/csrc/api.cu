// C-ABI entry points (include/optimobo_b200.h).  Plain pointers and sizes only.
#include <stdarg.h>
#include <stdlib.h>

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
    k.fast_mode = geti("OMBO_FAST_MODE", 0);
    k.fast_cluster = geti("OMBO_FAST_CLUSTER", 1);
    k.fast_dbg = geti("OMBO_FAST_DBG", 0);
    k.fast_profile = geti("OMBO_FAST_PROFILE", 0);
    k.fast_notrim = getenv("OMBO_FAST_NOTRIM") != nullptr;
    k.fast_nocache = getenv("OMBO_FAST_NOCACHE") != nullptr;
    k.fast_zerocache = getenv("OMBO_FAST_ZEROCACHE") != nullptr;
    k.fast_mean_in_main = getenv("OMBO_FAST_MEAN_IN_MAIN") != nullptr;
    k.fast_gen_warps = geti("OMBO_FAST_GEN_WARPS", 8);
    k.f8_max_run = geti("OMBO_F8_MAXRUN", 0);
    { const char *e = getenv("OMBO_F8_TG"); k.f8_tg = e ? atof(e) : 3.0; }
    k.chunk_log2 = geti("OMBO_CHUNK_LOG2", OMBO_CHUNK_DEV_LOG2);
    if (k.chunk_log2 < 10) k.chunk_log2 = 10;
    if (k.chunk_log2 > 26) k.chunk_log2 = 26;
    k.no_f8c = getenv("OMBO_NO_F8C") != nullptr;
    { const char *e = getenv("OMBO_F8C_KAPPA"); k.f8c_kappa = e ? atof(e) : OMBO_F8C_KAPPA_DEFAULT; }
    k.acq_fp64 = getenv("OMBO_ACQ_FP64") != nullptr;
    k.no_fuse = getenv("OMBO_NO_FUSE") != nullptr;
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
  if (c->f8_sched) cudaFree(c->f8_sched);
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

static int validate_score(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const ombo_acq *acq,
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
      OMBO_CHECK(k >= 2 && k <= OMBO_MAX_OBJ && n_gp >= k && acq->stripes && acq->cells,
                 "EHVI_BOX needs 2 <= n_obj <= %d, n_obj GPs, the breakpoint table and the boxes", OMBO_MAX_OBJ);
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

// scores rows [first, first+count) of the pool; X_dev points at row `first` (or NULL -> generator)
static int score_pass(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const void *X_dev,
                      long long first, long long count, const ombo_acq *acq, int precision, double *out_mu,
                      double *out_var, double *out_acq, long long out_ld, ombo_best *best_dev, cudaStream_t s) {
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
        case OMBO_ACQ_EHVI_BOX: want_var = (g < acq->n_obj); break;
        default: want_var = true;
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
                                       try_fuse ? &fq : nullptr, &fused);
    if (rc) return rc;
  }
  if (fused) return best_dev ? ombo_argmax_merge(ctx, fused, best_dev, s) : OMBO_OK;
  if (acq->kind != OMBO_ACQ_NONE)
    return ombo_acquire(ctx, acq, n_gp, mu, var, count, ld, pd.index_base, out_acq ? out_acq + first : nullptr,
                        best_dev, s, precision == OMBO_PREC_FAST);
  return OMBO_OK;
}

int ombo_score(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const ombo_acq *acq,
               int precision, double *out_mu, double *out_var, double *out_acq, ombo_best *best_dev,
               void *stream) {
  int rc = validate_score(ctx, gps, n_gp, pool, acq, precision);
  if (rc) return rc;
  OMBO_CHECK((out_mu == nullptr) == (out_var == nullptr), "score: out_mu and out_var must both be given or both NULL");
  OMBO_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (best_dev) { rc = ombo_best_init(ctx, best_dev, s); if (rc) return rc; }
  const size_t esz = pool->dtype == 0 ? 8 : 4;
  const long long chunk = 1LL << ctx->knobs.chunk_log2;
  for (long long first = 0; first < pool->m; first += chunk) {
    long long count = pool->m - first < chunk ? pool->m - first : chunk;
    const void *X = pool->X ? (const char *)pool->X + (size_t)first * pool->d * esz : nullptr;
    rc = score_pass(ctx, gps, n_gp, pool, X, first, count, acq, precision, out_mu, out_var, out_acq, pool->m,
                    best_dev, s);
    if (rc) return rc;
  }
  return OMBO_OK;
}

int ombo_score_host(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool, const ombo_acq *acq,
                    int precision, ombo_best *best_host, void *stream) {
  int rc = validate_score(ctx, gps, n_gp, pool, acq, precision);
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
    rc = score_pass(ctx, gps, n_gp, pool, X, first, count, acq, precision, nullptr, nullptr, nullptr, 0, best_dev, s);
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
  int rc = validate_score(ctx, gp_ok, n_gp, &fake, acq, OMBO_PREC_FP64);
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

int64_t ombo_launch_count(ombo_ctx *ctx, int reset) {
  if (!ctx) return 0;
  int64_t v = ctx->launches;
  if (reset) ctx->launches = 0;
  return v;
}

}  // extern "C"
