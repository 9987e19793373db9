// Stage 1 of the pruned arg-max (api.cu, score_pruned): the mean-only upper bound of the exact 2-D EHVI for both GPs
// of an f8c pair in one persistent launch.
//
// UB = ehvi2d_value<float>(mu0, mu1, var0_up, var1_up) with mu the full f8c launch's mean bit for bit and var_up the
// full launch's variance expression with sum V^2 = 0, i.e. fmax(sigma_f2, var_floor) + sigma_n2 >= var.  Over a valid
// front the exact EHVI never decreases in either sigma (DESIGN.md section 4), so UB bounds the candidate's value from
// above, like the chunk-0 bound of the BOUND launch but without any variance work.
//
// The training set of both GPs (scaled coordinates, sigma_f2 alpha, |b|^2: (DP + 2) floats per point) stays in shared
// memory for the whole launch: no slice ring, no TMA, no barrier inside the K loop, every warp a generator.  Warp
// (qq, rg) and lane map as the f8c generators: rows r16(lane) + 16 rr of the row group, column group g = 2 qq + (lane & 1);
// the K-blocks are walked in the order the full launch generates them (a table from f8_build_schedule) and the row is
// finished as there (lane-pair shuffle, then (p0 + p1) + (p2 + p3) over the four column pairs), with the arithmetic
// of gen8.cuh: mu is the full launch's FP32 mean.
#include <algorithm>
#include <vector>

#include "acq_math.cuh"
#include "gen8.cuh"

#define M8_WARPS 16                          // 4 column quarters x 4 row groups
#define M8_R 4                               // rows per lane
#define M8_TILE (M8_WARPS / 4 * 16 * M8_R)   // 256 candidates per tile
#define M8_MAX_KB (OMBO_MAX_TRAIN / 64)

struct Mean8Gp {
  const float *xs32, *alpha32, *b2_32;
  const double *ell, *center;       // device, (d) each
  int nkb;
  float var_up;
  unsigned char order[M8_MAX_KB];   // K-blocks in the order the full launch generates them
};

struct Mean8Params {
  Mean8Gp gp[2];
  PoolDev pool;
  long long m;
  int d, n_pf;
  float c00, c01;
  const double *stripes;            // 2 (n_pf + 2) doubles
  double *ub;                       // [m]: the bound as a double (NaN kept, as the fused epilogue's out_acq)
  double *mu_out;                   // optional [2][m]: the FP32 means as doubles (tests)
  ombo_best *partials;              // [gridDim.x] per-CTA (largest bound, global index)
};

// the K loop of one GP over the tile: this lane's share of the mean of its M8_R rows, into mub[qq][row]
template <int DP, bool MATERN>
__device__ __forceinline__ void mean8_gp(const Mean8Gp &g, const float *train, const float *xcg, float *mub, int qq,
                                         int row0, int gbit) {
  constexpr int XT = (DP + 2) * 64;
  float x[M8_R][DP], a2[M8_R], mu_acc[M8_R];
#pragma unroll
  for (int rr = 0; rr < M8_R; ++rr) {
    mu_acc[rr] = 0.f;
    a2[rr] = gen8_load_row<DP>(xcg + row0 + 16 * rr, M8_TILE, x[rr]);
  }
  const int col = 8 * (2 * qq + gbit);
#pragma unroll 1
  for (int s = 0; s < g.nkb; ++s) {
    const float *xs = train + (size_t)g.order[s] * XT + col;
    float2 r2[M8_R][4];
    gen8_dist2<DP, M8_R>(xs, x, a2, r2);
    const float4 al0 = *(const float4 *)(xs + DP * 64);
    const float4 al1 = *(const float4 *)(xs + DP * 64 + 4);
#pragma unroll
    for (int rr = 0; rr < M8_R; ++rr) {
      float2 kv[4];
      gen8_kval<MATERN>(r2[rr], kv);
      gen8_mean_add(kv, al0, al1, mu_acc[rr]);
    }
  }
#pragma unroll
  for (int rr = 0; rr < M8_R; ++rr) {
    const float m = mu_acc[rr] + __shfl_xor_sync(0xffffffffu, mu_acc[rr], 1);
    if (!gbit) mub[qq * M8_TILE + row0 + 16 * rr] = m;
  }
}

template <int DP, bool MAT0, bool MAT1>
__global__ void __launch_bounds__(M8_WARPS * 32, 1) k_posterior_mean8(const __grid_constant__ Mean8Params p) {
  extern __shared__ __align__(16) float m8_smem[];
  constexpr int XT = (DP + 2) * 64;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nt = M8_WARPS * 32;
  float *train0 = m8_smem;                                        // [nkb][DP + 2][64] per GP
  float *train1 = train0 + (size_t)p.gp[0].nkb * XT;
  float *xc = train1 + (size_t)p.gp[1].nkb * XT;                  // [2][DP][M8_TILE] scaled coordinates of the tile
  float *mub = xc + 2 * DP * M8_TILE;                             // [2][4][M8_TILE] column-pair partials of the mean
  float *ystr = mub + 8 * M8_TILE;                                // [2 (n_pf + 2)] stripe bounds in FP32
  double *red_v = (double *)(((uintptr_t)(ystr + 2 * (p.n_pf + 2)) + 15) & ~(uintptr_t)15);
  long long *red_i = (long long *)(red_v + M8_WARPS);
  double *geo = (double *)(red_i + M8_WARPS);                     // [2][centre (12), 1 / ell (12)]

  for (int gi = 0; gi < 2; ++gi) {
    const Mean8Gp &g = p.gp[gi];
    float *t = gi ? train1 : train0;
    const int np = g.nkb * 64;
    for (int e = tid; e < g.nkb * XT; e += nt) {
      const int kb = e / XT, r = e % XT, jj = r >> 6, c = kb * 64 + (r & 63);
      t[e] = jj < DP ? g.xs32[(size_t)jj * np + c] : (jj == DP ? g.alpha32[c] : g.b2_32[c]);
    }
  }
  for (int i = tid; i < 2 * (p.n_pf + 2); i += nt) ystr[i] = (float)p.stripes[i];
  if (tid < 24) {                                                 // as k_posterior_fast8 derives them
    const int gi = tid / 12, j = tid % 12;
    geo[gi * 24 + j] = j < p.d ? p.gp[gi].center[j] : 0.0;
    geo[gi * 24 + 12 + j] = j < p.d ? 1.0 / p.gp[gi].ell[j] : 0.0;
  }
  for (int e = tid; e < 2 * DP * M8_TILE; e += nt) xc[e] = 0.f;     // dimensions >= d stay 0
  __syncthreads();

  const int qq = warp & 3, rg = warp >> 2, gbit = lane & 1;
  const int r16 = ((lane >> 1) & 3) * 2 + ((lane >> 3) & 1) + 8 * (lane >> 4);
  const int row0 = 16 * M8_R * rg + r16;
  const long long n_tiles = (p.m + M8_TILE - 1) / M8_TILE;
  BestPair best;
  best.v = -INFINITY; best.i = 0x7fffffffffffffffLL;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    // coordinates of the tile for both GPs (one pool read per coordinate); the previous tile's readers of xc have
    // passed the barrier behind their K loops
    for (int e = tid; e < p.d * M8_TILE; e += nt) {
      const int r = e % M8_TILE, j = e / M8_TILE;
      const long long cg = tile * M8_TILE + r;
      float x0 = 0.f, x1 = 0.f;
      if (cg < p.m) {
        const double a = ombo_pool_coord(p.pool, cg, j);
        x0 = gen8_coord(a, geo[j], geo[12 + j]);
        x1 = gen8_coord(a, geo[24 + j], geo[36 + j]);
      }
      xc[j * M8_TILE + r] = x0;
      xc[(DP + j) * M8_TILE + r] = x1;
    }
    __syncthreads();
    mean8_gp<DP, MAT0>(p.gp[0], train0, xc, mub, qq, row0, gbit);
    mean8_gp<DP, MAT1>(p.gp[1], train1, xc + DP * M8_TILE, mub + 4 * M8_TILE, qq, row0, gbit);
    __syncthreads();
    if (tid < M8_TILE) {
      const long long cg = tile * M8_TILE + tid;
      const float mu0 = gen8_mean_sum(mub[tid], mub[M8_TILE + tid], mub[2 * M8_TILE + tid], mub[3 * M8_TILE + tid]);
      const float *m1 = mub + 4 * M8_TILE;
      const float mu1 = gen8_mean_sum(m1[tid], m1[M8_TILE + tid], m1[2 * M8_TILE + tid], m1[3 * M8_TILE + tid]);
      if (cg < p.m) {
        const int P = p.n_pf;
        const float r = ehvi2d_value<float>(mu0, mu1, p.gp[0].var_up, p.gp[1].var_up, ystr, ystr + (P + 2), P, true,
                                            p.c00, p.c01);
        p.ub[cg] = (double)r;
        if (p.mu_out) { p.mu_out[cg] = (double)mu0; p.mu_out[p.m + cg] = (double)mu1; }
        const double val = isnan(r) ? -INFINITY : (double)r;
        const long long gi = p.pool.index_base + cg;
        if (better(val, gi, best.v, best.i)) { best.v = val; best.i = gi; }
      }
    }
  }
  best = warp_best(best);
  if (lane == 0) { red_v[warp] = best.v; red_i[warp] = best.i; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < M8_WARPS; ++w)
      if (better(red_v[w], red_i[w], best.v, best.i)) { best.v = red_v[w]; best.i = red_i[w]; }
    p.partials[blockIdx.x].value = best.v;
    p.partials[blockIdx.x].index = best.i;
  }
}

void f8_build_schedule(int np, double tg, int max_run, std::vector<unsigned int> &steps, int bound_chunks);

static size_t mean8_smem(int dp, int nkb0, int nkb1, int n_pf) {
  return ((size_t)(nkb0 + nkb1) * (dp + 2) * 64 + 2 * (size_t)dp * M8_TILE + 8 * M8_TILE + 2 * (size_t)(n_pf + 2)) * 4 +
         16 + (size_t)M8_WARPS * 16 + 2 * 24 * 8;
}

static int mean8_dp(int d) { return d <= 2 ? 2 : (d + 1) / 2 * 2; }

bool ombo_mean8_covers(const GpDev gp[2], int n_pf) {
  const int d = gp[0].d;
  return d <= 12 && gp[1].d == d && mean8_smem(mean8_dp(d), gp[0].n_pad / 64, gp[1].n_pad / 64, n_pf) <= 227 * 1024;
}

template <int DP, bool MAT0, bool MAT1>
static int launch_mean8(const Mean8Params &p, size_t smem, int grid, cudaStream_t s) {
  OMBO_CUDA(cudaFuncSetAttribute(k_posterior_mean8<DP, MAT0, MAT1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_posterior_mean8<DP, MAT0, MAT1><<<grid, M8_WARPS * 32, smem, s>>>(p);
  OMBO_CUDA(cudaGetLastError());
  return OMBO_OK;
}

int ombo_mean8_bound(ombo_ctx *ctx, const GpDev gp[2], const PoolDev &pool, long long m, const double *stripes,
                     int n_pf, float c00, float c01, double *ub, ombo_best *best_dev, double *mu_out, int *grid_out,
                     cudaStream_t s) {
  if (!ombo_mean8_covers(gp, n_pf)) { ombo_set_error("mean8: shape not covered"); return OMBO_ERR_UNSUPPORTED; }
  Mean8Params p;
  memset(&p, 0, sizeof(p));
  for (int g = 0; g < 2; ++g) {
    Mean8Gp &q = p.gp[g];
    q.xs32 = gp[g].xs32; q.alpha32 = gp[g].alpha32; q.b2_32 = gp[g].b2_32;
    q.nkb = gp[g].n_pad / 64;
    // the full launch's variance with sum V^2 = 0 (its epilogue: fmax(sigma_f2 - ss / s^2, floor) + sigma_n2)
    q.var_up = (float)(fmax(gp[g].sigma_f2, gp[g].var_floor) + gp[g].sigma_n2);
    q.ell = gp[g].ell; q.center = gp[g].center;
    std::vector<unsigned int> steps;
    f8_build_schedule(gp[g].n_pad, ctx->knobs.f8_tg, ctx->knobs.f8_max_run, steps, 0);
    int n = 0;
    for (unsigned int w : steps)
      if ((w >> 8) & 1u) q.order[n++] = (unsigned char)(w & 0xFFu);
    if (n != q.nkb) { ombo_set_error("mean8: schedule has %d fresh blocks, expected %d", n, q.nkb); return OMBO_ERR_CUDA; }
  }
  p.pool = pool; p.m = m; p.d = gp[0].d; p.n_pf = n_pf; p.c00 = c00; p.c01 = c01;
  p.stripes = stripes; p.ub = ub; p.mu_out = mu_out;
  const long long tiles = (m + M8_TILE - 1) / M8_TILE;
  const int grid = (int)std::max(1LL, std::min(tiles, (long long)ctx->num_sms));
  if (grid_out) *grid_out = grid;
  int rc = ombo_ws_reserve(&ctx->ws_partial, &ctx->ws_partial_bytes, (size_t)grid * sizeof(ombo_best));
  if (rc) return rc;
  p.partials = (ombo_best *)ctx->ws_partial;
  const int dp = mean8_dp(p.d);
  const size_t smem = mean8_smem(dp, p.gp[0].nkb, p.gp[1].nkb, n_pf);
  const bool m0 = gp[0].kernel == OMBO_KERNEL_MATERN52, m1 = gp[1].kernel == OMBO_KERNEL_MATERN52;
  {
    ProfScope prof(ctx, s);
#define M8_LAUNCH(DPV)                                                                                               \
  rc = m0 ? (m1 ? launch_mean8<DPV, true, true>(p, smem, grid, s) : launch_mean8<DPV, true, false>(p, smem, grid, s))  \
          : (m1 ? launch_mean8<DPV, false, true>(p, smem, grid, s) : launch_mean8<DPV, false, false>(p, smem, grid, s))
    if (dp == 2) { M8_LAUNCH(2); }
    else if (dp == 4) { M8_LAUNCH(4); }
    else if (dp == 6) { M8_LAUNCH(6); }
    else if (dp == 8) { M8_LAUNCH(8); }
    else if (dp == 10) { M8_LAUNCH(10); }
    else { M8_LAUNCH(12); }
#undef M8_LAUNCH
  }
  if (rc) return rc;
  ctx->launches += 1;
  return ombo_argmax_merge(ctx, grid, best_dev, s);
}
