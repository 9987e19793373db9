// Box decomposition of the region no front point dominates, for the exact EHVI of 2 <= k <= 4 objectives
// (ombo_ehvi_boxes): the device twin of host_prep.ehvi_boxes, equal to it element for element and in its order.
//
// Everything is done in breakpoint-index ("rank") space.  Every corner host_prep.ehvi_boxes produces is -inf, a front
// coordinate of its objective or r_i, and searchsorted(row_i, v, "left") = 1 + #{distinct front values of objective i
// < v} for finite v, 0 for -inf.  Ranks keep the order of the values, so dominance and "first front" can be decided on
// ranks, and the ranks are the output.
//
// The host recursion, written out for k = 4 (for k = 3 drop the j4 level, for k = 2 the j3 level too):
//   j4 in [0, m4]: E4 = rank j4 (0 = -inf), U4 = j4 + 1 or the rank of r_3; skipped when U4 <= E4;
//     sub3(j4) = 3-D front of {p : rank4(p) <= E4};  L(j4) = its distinct objective-3 ranks, ascending;
//     j3 in [0, |L|]: E3 = L[j3 - 1] (0 for j3 = 0), U3 = L[j3] or the rank of r_2; skipped when U3 <= E3;
//       the 2-D staircase of {p : rank4(p) <= E4, rank3(p) <= E3} projected on objectives 1, 2: b_1 < ... < b_n with
//       a_1 > ... > a_n; box j2 in [0, n] = lower (0, b_j2, E3, E4), upper (a_j2, b_j2+1, U3, U4) with a_0 = rank(r_0),
//       b_0 = 0, b_n+1 = rank(r_1); the last is skipped when b_n = rank(r_1).
// Two facts make this cheap.  (1) The 2-D front of the sub-front's points with rank3 <= E3 has the same points as the
// 2-D front of ALL front points with rank4 <= E4 and rank3 <= E3: a point the 3-D front drops is weakly dominated by
// one it keeps, which passes the same filter.  (2) A point p belongs to sub3(j4) exactly for rank4(p) <= j4 < d(p),
// d(p) = least rank4 of the points that dominate p in objectives 1..3 (they all have rank4 > rank4(p), p being on the
// 4-D front).  So L(j4) is one pass over the points per j4, and each (j4, j3) tuple is an independent warp job.
//
// Passes: k_box_front (first front, duplicates, filter; many blocks) -> k_box_table (ranks, table, L(j4), the tuple
// list; one block) -> k_box_tuples<false> (boxes per tuple) -> inclusive scan -> one read-back -> k_box_tuples<true>.
#include <cub/block/block_scan.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace {

constexpr int BX_MAX_PTS = OMBO_EHVI_BOX_MAX_BREAKS - 2;   // 512 distinct front points
constexpr int BX_LD = BX_MAX_PTS;                          // row stride of the L(j4) lists
constexpr int BX_TABLE_THREADS = 1024;
constexpr int BX_TUPLE_WARPS = 8;
constexpr int BX_BIG = 0x7fffffff;

enum { BX_OK = 0, BX_NEG_INF = 1, BX_TOO_MANY = 2 };

// r_c without a local-memory array
__device__ __forceinline__ double ref_c(int c, double r0, double r1, double r2, double r3) {
  return c == 0 ? r0 : c == 1 ? r1 : c == 2 ? r2 : r3;
}

struct BoxHdr {
  int status;        // BX_*
  int u;             // distinct front points
  int B;             // breakpoints per objective
  int n_out;         // level-4 slices (1 for k <= 3)
  int n_tuples;      // (j4, j3) jobs
  int m[4];          // distinct values per objective
  int rr[4];         // breakpoint index of r_i
  int neg_inf;       // set by k_box_front: a row inside r has a -inf coordinate
};
static_assert(sizeof(BoxHdr) + sizeof(int) <= 64, "BoxHdr and the box count are read back through the 64-byte pinned buffer");

// flag[j] = 1 when row j is <= r, on the first front (no row is <= it everywhere and < somewhere) and no earlier row is
// identical.  Rows beyond r or with a NaN never dominate a row <= r, so the sweep needs no filter on i.
__global__ void k_box_front(const double *__restrict__ Y, int n, int k, double r0, double r1, double r2, double r3,
                            unsigned char *__restrict__ flag, BoxHdr *__restrict__ hdr) {
  extern __shared__ double tile[];               // (blockDim.x, k) rows of the sweep
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  double yj[4] = {0.0, 0.0, 0.0, 0.0};
  bool keep = j < n, ninf = false;
#pragma unroll
  for (int c = 0; c < 4; ++c)
    if (c < k) {
      yj[c] = j < n ? Y[(size_t)j * k + c] : 0.0;
      keep = keep && yj[c] <= ref_c(c, r0, r1, r2, r3);
      ninf = ninf || yj[c] == -INFINITY;
    }
  if (keep && ninf) atomicOr(&hdr->neg_inf, 1);
  bool drop = !keep;
  for (int i0 = 0; i0 < n; i0 += blockDim.x) {
    const int rows = min((int)blockDim.x, n - i0);
    for (int e = threadIdx.x; e < rows * k; e += blockDim.x) tile[e] = Y[(size_t)i0 * k + e];
    __syncthreads();
    if (!drop) {
      for (int ii = 0; ii < rows; ++ii) {
        bool le = true, lt = false, eq = true;
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (c < k) {
            const double v = tile[ii * k + c];
            le = le && (v <= yj[c]);
            lt = lt || (v < yj[c]);
            eq = eq && (v == yj[c]);
          }
        if ((le && lt) || (eq && i0 + ii < j)) { drop = true; break; }
      }
    }
    __syncthreads();
  }
  if (j < n) flag[j] = drop ? 0 : 1;
}

// One block.  Gathers the u flagged rows, ranks them, writes the (k, B) table to table_ws, the lists L(j4) and the
// tuple list tup[t] = (j4 << 16) | j3 in lexicographic order.
__global__ void __launch_bounds__(BX_TABLE_THREADS, 1)
k_box_table(const double *__restrict__ Y, int n, int k, double r0, double r1, double r2, double r3,
            const unsigned char *__restrict__ flag, BoxHdr *__restrict__ hdr, ushort4 *__restrict__ rk,
            unsigned short *__restrict__ L, int *__restrict__ mL, unsigned int *__restrict__ tup,
            double *__restrict__ table_ws) {
  using Scan = cub::BlockScan<int, BX_TABLE_THREADS>;
  __shared__ typename Scan::TempStorage scan_tmp;
  __shared__ int idx[BX_MAX_PTS];
  __shared__ double F[BX_MAX_PTS][4];
  __shared__ unsigned short R[BX_MAX_PTS][4];
  __shared__ unsigned short dlim[BX_MAX_PTS];
  __shared__ unsigned char first[BX_MAX_PTS][4];
  __shared__ int ns[BX_MAX_PTS + 1];
  __shared__ unsigned int bits[BX_TABLE_THREADS / 32][(BX_MAX_PTS + 1 + 31) / 32];
  __shared__ int m_s[4], rr_s[4];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // ---- gather the flagged rows (any order would do: everything below depends on values only)
  const int per = (n + BX_TABLE_THREADS - 1) / BX_TABLE_THREADS;
  const int a0 = min(n, tid * per), a1 = min(n, a0 + per);
  int cnt = 0;
  for (int j = a0; j < a1; ++j) cnt += flag[j];
  int pos, total;
  Scan(scan_tmp).ExclusiveSum(cnt, pos, total);
  for (int j = a0; j < a1; ++j)
    if (flag[j]) { if (pos < BX_MAX_PTS) idx[pos] = j; ++pos; }
  if (tid < 4) { m_s[tid] = 0; rr_s[tid] = 1; }
  __syncthreads();
  if (hdr->neg_inf || total > BX_MAX_PTS) {
    if (tid == 0) {
      hdr->status = hdr->neg_inf ? BX_NEG_INF : BX_TOO_MANY;
      hdr->u = total; hdr->B = 0; hdr->n_out = 0; hdr->n_tuples = 0;
    }
    return;
  }
  const int u = total;
  for (int e = tid; e < u * 4; e += BX_TABLE_THREADS) {
    const int p = e >> 2, c = e & 3;
    F[p][c] = c < k ? Y[(size_t)idx[p] * k + c] : 0.0;
  }
  __syncthreads();
  // ---- ranks: first occurrence of each value per objective, then 1 + #{distinct values below}
  for (int e = tid; e < u * 4; e += BX_TABLE_THREADS) {
    const int p = e >> 2, c = e & 3;
    bool f = c < k;
    for (int q = 0; q < p && f; ++q) f = F[q][c] != F[p][c];
    first[p][c] = f;
  }
  __syncthreads();
  for (int e = tid; e < u * 4; e += BX_TABLE_THREADS) {
    const int p = e >> 2, c = e & 3;
    int below = 0;
    if (c < k)
      for (int q = 0; q < u; ++q) below += first[q][c] && F[q][c] < F[p][c];
    R[p][c] = c < k ? (unsigned short)(1 + below) : 0;
    if (first[p][c]) atomicAdd(&m_s[c], 1);
  }
  for (int e = tid; e < 4 * 32; e += BX_TABLE_THREADS) {     // rank of r_c: 1 + #{distinct values < r_c}
    const int c = e >> 5;
    int below = 0;
    if (c < k)
      for (int q = e & 31; q < u; q += 32) below += first[q][c] && F[q][c] < ref_c(c, r0, r1, r2, r3);
    for (int o = 16; o; o >>= 1) below += __shfl_xor_sync(0xffffffffu, below, o);
    if ((e & 31) == 0 && c < k) rr_s[c] = 1 + below;
  }
  __syncthreads();
  int B = 0;
  for (int c = 0; c < k; ++c) B = max(B, m_s[c] + 2);
  // ---- table row c = [-inf, sorted distinct values, r_c, padded with r_c]
  for (int e = tid; e < k * B; e += BX_TABLE_THREADS) {
    const int c = e / B, i = e % B;
    if (i == 0) table_ws[e] = -INFINITY;
    else if (i > m_s[c]) table_ws[e] = ref_c(c, r0, r1, r2, r3);
  }
  for (int e = tid; e < u * 4; e += BX_TABLE_THREADS) {
    const int p = e >> 2, c = e & 3;
    if (c < k && first[p][c]) table_ws[c * B + R[p][c]] = F[p][c];
  }
  // ---- d(p): least rank4 among the points that dominate p in objectives 1..3 (65535: none; always none for k <= 3)
  for (int p = tid; p < u; p += BX_TABLE_THREADS) {
    int d = 0xffff;
    for (int q = 0; q < u; ++q) {
      const bool le = R[q][0] <= R[p][0] && R[q][1] <= R[p][1] && R[q][2] <= R[p][2];
      const bool lt = R[q][0] < R[p][0] || R[q][1] < R[p][1] || R[q][2] < R[p][2];
      if (le && lt) d = min(d, (int)R[q][3]);
    }
    dlim[p] = (unsigned short)d;
    rk[p] = make_ushort4(R[p][0], R[p][1], R[p][2], R[p][3]);
  }
  __syncthreads();
  // level-4 slices: j4 = m_3 is empty when t_m4 = r_3 (its rank is then m_3)
  const int n_out = k == 4 ? m_s[3] + 1 - (rr_s[3] == m_s[3] ? 1 : 0) : 1;
  // ---- L(j4) = distinct objective-3 ranks of {p : rank4(p) <= j4 < d(p)}, one warp per j4
  constexpr int W = (BX_MAX_PTS + 1 + 31) / 32;
  for (int o = warp; o < n_out; o += BX_TABLE_THREADS / 32) {
    if (lane < W) bits[warp][lane] = 0u;
    __syncwarp();
    for (int p = lane; p < u; p += 32) {
      const int z = R[p][2];
      if (z >= 1 && R[p][3] <= o && o < dlim[p]) atomicOr(&bits[warp][z >> 5], 1u << (z & 31));
    }
    __syncwarp();
    const unsigned int w = lane < W ? bits[warp][lane] : 0u;
    int c = __popc(w), off = c;
    for (int s = 1; s < 32; s <<= 1) { const int v = __shfl_up_sync(0xffffffffu, off, s); if (lane >= s) off += v; }
    const int m = __shfl_sync(0xffffffffu, off, 31);
    off -= c;
    for (unsigned int x = w; x; x &= x - 1) L[(size_t)o * BX_LD + off++] = (unsigned short)(lane * 32 + __ffs(x) - 1);
    __syncwarp();
    if (lane == 0) {
      mL[o] = m;
      // j3 = m is empty when the top value of the sub-front equals r_2
      ns[o] = m + 1 - (m >= 1 && L[(size_t)o * BX_LD + m - 1] == rr_s[2] ? 1 : 0);
    }
  }
  __syncthreads();
  // ---- the tuple list in (j4, j3) order
  const int my = tid < n_out ? ns[tid] : 0;
  int base, n_tuples;
  Scan(scan_tmp).ExclusiveSum(my, base, n_tuples);
  for (int j3 = 0; j3 < my; ++j3) tup[base + j3] = ((unsigned int)tid << 16) | (unsigned int)j3;
  if (tid == 0) {
    hdr->status = BX_OK; hdr->u = u; hdr->B = B; hdr->n_out = n_out; hdr->n_tuples = n_tuples;
    for (int c = 0; c < 4; ++c) { hdr->m[c] = m_s[c]; hdr->rr[c] = rr_s[c]; }
  }
}

// One warp per (j4, j3) tuple.  EMIT = false: cnt[t] = boxes of tuple t (0 for t >= n_tuples, up to n_slots).
// EMIT = true: writes tuple t's boxes from offs[t] - cnt[t] on, as f64 indices in the (n_boxes, 2, k) layout.
template <bool EMIT>
__global__ void __launch_bounds__(BX_TUPLE_WARPS * 32, 4)
k_box_tuples(const BoxHdr *__restrict__ hdr, int k, const ushort4 *__restrict__ rk,
             const unsigned short *__restrict__ L, const int *__restrict__ mL, const unsigned int *__restrict__ tup,
             int *__restrict__ cnt, const int *__restrict__ offs, int n_slots, double *__restrict__ boxes) {
  __shared__ ushort4 pts[BX_MAX_PTS];
  __shared__ int minA[BX_TUPLE_WARPS][BX_MAX_PTS + 2];
  __shared__ unsigned short fa[EMIT ? BX_TUPLE_WARPS : 1][BX_MAX_PTS + 2], fb[EMIT ? BX_TUPLE_WARPS : 1][BX_MAX_PTS + 2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int u = hdr->u, n_tuples = hdr->n_tuples, m1 = hdr->m[1], m3 = hdr->m[3];
  const int rr0 = hdr->rr[0], rr1 = hdr->rr[1], rr2 = hdr->rr[2], rr3 = hdr->rr[3];
  for (int p = threadIdx.x; p < u && n_tuples > 0; p += blockDim.x) pts[p] = rk[p];
  __syncthreads();
  const int chunk = (m1 + 31) / 32, b0 = 1 + lane * chunk, b1 = min(b0 + chunk, m1 + 1);
  const int stride = gridDim.x * BX_TUPLE_WARPS;
  const int t_end = EMIT ? n_tuples : n_slots;
  for (int t = blockIdx.x * BX_TUPLE_WARPS + warp; t < t_end; t += stride) {
    if (!EMIT && t >= n_tuples) { if (lane == 0) cnt[t] = 0; continue; }
    const unsigned int tv = tup[t];
    const int o = (int)(tv >> 16), j3 = (int)(tv & 0xffffu), mo = mL[o];
    const int E4 = k == 4 ? o : 0, U4 = o < m3 ? o + 1 : rr3;
    const int E3 = j3 == 0 ? 0 : L[(size_t)o * BX_LD + j3 - 1];
    const int U3 = j3 < mo ? L[(size_t)o * BX_LD + j3] : rr2;
    int *mA = minA[warp];
    for (int b = 1 + lane; b <= m1; b += 32) mA[b] = BX_BIG;
    __syncwarp();
    for (int p = lane; p < u; p += 32) {
      const ushort4 q = pts[p];
      if (q.w <= E4 && q.z <= E3) atomicMin(&mA[q.y], (int)q.x);
    }
    __syncwarp();
    // staircase on objective 2: b is a step when its least objective-1 rank is below every earlier one
    int lmin = BX_BIG;
    for (int b = b0; b < b1; ++b) lmin = min(lmin, mA[b]);
    for (int s = 1; s < 32; s <<= 1) { const int v = __shfl_up_sync(0xffffffffu, lmin, s); if (lane >= s) lmin = min(lmin, v); }
    int run = __shfl_up_sync(0xffffffffu, lmin, 1);
    if (lane == 0) run = BX_BIG;
    const int run0 = run;
    int c = 0, last = 0;
    for (int b = b0; b < b1; ++b) { const int v = mA[b]; if (v < run) { ++c; run = v; last = b; } }
    int off = c;
    for (int s = 1; s < 32; s <<= 1) { const int v = __shfl_up_sync(0xffffffffu, off, s); if (lane >= s) off += v; }
    const int nst = __shfl_sync(0xffffffffu, off, 31);
    for (int s = 16; s; s >>= 1) last = max(last, __shfl_xor_sync(0xffffffffu, last, s));
    const int count = nst + 1 - (nst >= 1 && last == rr1 ? 1 : 0);
    if (!EMIT) {
      if (lane == 0) cnt[t] = count;
    } else {
      unsigned short *A = fa[warp], *Bq = fb[warp];
      off -= c;
      run = run0;
      for (int b = b0; b < b1; ++b) {
        const int v = mA[b];
        if (v < run) { run = v; ++off; A[off] = (unsigned short)v; Bq[off] = (unsigned short)b; }
      }
      if (lane == 0) { A[0] = (unsigned short)rr0; Bq[0] = 0; Bq[nst + 1] = (unsigned short)rr1; }
      __syncwarp();
      const long long first_box = (long long)offs[t] - count;
      for (int j2 = lane; j2 < count; j2 += 32) {
        double *out = boxes + (size_t)(first_box + j2) * 2 * k;
        out[0] = (double)A[j2];
        out[1] = (double)Bq[j2 + 1];
        out[k] = 0.0;
        out[k + 1] = (double)Bq[j2];
        if (k >= 3) { out[2] = (double)U3; out[k + 2] = (double)E3; }
        if (k == 4) { out[3] = (double)U4; out[k + 3] = (double)E4; }
      }
    }
    __syncwarp();
  }
}

}  // namespace

int ombo_ehvi_boxes_impl(ombo_ctx *ctx, const double *PF, int p, int k, const double *ref, double *table,
                         double *boxes, long long boxes_cap, int *B_out, long long *n_boxes_out, cudaStream_t s) {
  const int pu = min(p, BX_MAX_PTS);
  const int n_slots = k == 4 ? (pu + 1) * (pu + 1) : k == 3 ? pu + 1 : 1;   // bound on the (j4, j3) tuples
  size_t cub_bytes = 0;
  OMBO_CUDA(cub::DeviceScan::InclusiveSum(nullptr, cub_bytes, (const int *)nullptr, (int *)nullptr, n_slots, s));
  auto al = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t o_flag = al(sizeof(BoxHdr)), o_rk = o_flag + al((size_t)max(p, 1));
  const size_t o_L = o_rk + al(sizeof(ushort4) * BX_MAX_PTS);
  const size_t o_mL = o_L + al(sizeof(unsigned short) * (size_t)(BX_MAX_PTS + 1) * BX_LD);
  const size_t o_tup = o_mL + al(sizeof(int) * (BX_MAX_PTS + 1));
  const size_t o_cnt = o_tup + al(sizeof(unsigned int) * (size_t)n_slots);
  const size_t o_offs = o_cnt + al(sizeof(int) * (size_t)n_slots);
  const size_t o_table = o_offs + al(sizeof(int) * (size_t)n_slots);
  const size_t o_cub = o_table + al(sizeof(double) * 4 * (BX_MAX_PTS + 2));
  int rc = ombo_ws_reserve(&ctx->ws_boxprep, &ctx->ws_boxprep_bytes, o_cub + cub_bytes);
  if (rc) return rc;
  char *ws = (char *)ctx->ws_boxprep;
  BoxHdr *hdr = (BoxHdr *)ws;
  unsigned char *flag = (unsigned char *)(ws + o_flag);
  ushort4 *rk = (ushort4 *)(ws + o_rk);
  unsigned short *L = (unsigned short *)(ws + o_L);
  int *mL = (int *)(ws + o_mL), *cnt = (int *)(ws + o_cnt), *offs = (int *)(ws + o_offs);
  unsigned int *tup = (unsigned int *)(ws + o_tup);
  double *table_ws = (double *)(ws + o_table);
  const double r[4] = {ref[0], ref[1], k > 2 ? ref[2] : 0.0, k > 3 ? ref[3] : 0.0};

  OMBO_CUDA(cudaMemsetAsync(hdr, 0, sizeof(BoxHdr), s));
  if (p > 0) {
    const int threads = 256;
    k_box_front<<<(p + threads - 1) / threads, threads, (size_t)threads * k * sizeof(double), s>>>(
        PF, p, k, r[0], r[1], r[2], r[3], flag, hdr);
    OMBO_CUDA(cudaGetLastError());
  }
  k_box_table<<<1, BX_TABLE_THREADS, 0, s>>>(PF, p, k, r[0], r[1], r[2], r[3], flag, hdr, rk, L, mL, tup, table_ws);
  OMBO_CUDA(cudaGetLastError());
  const int grid = max(1, min((n_slots + BX_TUPLE_WARPS - 1) / BX_TUPLE_WARPS, ctx->num_sms * 8));
  k_box_tuples<false><<<grid, BX_TUPLE_WARPS * 32, 0, s>>>(hdr, k, rk, L, mL, tup, cnt, nullptr, n_slots, nullptr);
  OMBO_CUDA(cudaGetLastError());
  OMBO_CUDA(cub::DeviceScan::InclusiveSum(ws + o_cub, cub_bytes, cnt, offs, n_slots, s));
  ctx->launches += (p > 0 ? 1 : 0) + 3;
  // the call's one synchronise: the header and the box count
  OMBO_CUDA(cudaMemcpyAsync(ctx->pinned_best, hdr, sizeof(BoxHdr), cudaMemcpyDeviceToHost, s));
  OMBO_CUDA(cudaMemcpyAsync((char *)ctx->pinned_best + sizeof(BoxHdr), offs + n_slots - 1, sizeof(int),
                            cudaMemcpyDeviceToHost, s));
  OMBO_CUDA(cudaStreamSynchronize(s));
  BoxHdr h;
  int n_boxes;
  memcpy(&h, ctx->pinned_best, sizeof(BoxHdr));
  memcpy(&n_boxes, (char *)ctx->pinned_best + sizeof(BoxHdr), sizeof(int));
  *B_out = 0;
  *n_boxes_out = 0;
  if (h.status == BX_NEG_INF) {
    ombo_set_error("ehvi_boxes: a row inside the reference point has a -inf coordinate");
    return OMBO_ERR_INVALID;
  }
  if (h.status == BX_TOO_MANY) {
    ombo_set_error("ehvi_boxes: the first front has %d distinct points inside the reference point, supported up to %d",
                   h.u, BX_MAX_PTS);
    return OMBO_ERR_UNSUPPORTED;
  }
  *B_out = h.B;
  *n_boxes_out = n_boxes;
  if (h.B > OMBO_EHVI_BOX_MAX_BREAKS) {
    ombo_set_error("ehvi_boxes: %d breakpoints per objective, the box EHVI takes up to %d", h.B,
                   OMBO_EHVI_BOX_MAX_BREAKS);
    return OMBO_ERR_INVALID;
  }
  if (n_boxes > OMBO_EHVI_BOX_MAX_BOXES) {
    ombo_set_error("ehvi_boxes: the decomposition has %d boxes, the box EHVI takes up to %d", n_boxes,
                   OMBO_EHVI_BOX_MAX_BOXES);
    return OMBO_ERR_INVALID;
  }
  if (n_boxes > boxes_cap) {
    ombo_set_error("ehvi_boxes: the decomposition has %d boxes, the buffer holds %lld", n_boxes, boxes_cap);
    return OMBO_ERR_SPACE;
  }
  OMBO_CUDA(cudaMemcpyAsync(table, table_ws, sizeof(double) * (size_t)k * h.B, cudaMemcpyDeviceToDevice, s));
  k_box_tuples<true><<<grid, BX_TUPLE_WARPS * 32, 0, s>>>(hdr, k, rk, L, mL, tup, cnt, offs, n_slots, boxes);
  OMBO_CUDA(cudaGetLastError());
  ctx->launches += 1;
  return OMBO_OK;
}
