// Exact top-k of the acquisition over a whole device pool (ombo_score_topk).
//
// Every pass of the pool (2^OMBO_CHUNK_LOG2 candidates) runs through the same ombo_score_pass as ombo_score, with
// out_acq pointed at a workspace of the pass size, so the values are the ones ombo_score writes (fused f8c epilogue,
// k_acquire, k_acquire_box).  The pass is then merged into a running k-list kept on the device:
//   1. keys: each value maps to an order-preserving 64-bit key (NaN -> -inf, -0 -> +0, as a comparison ranks them);
//      the running list's keys go in front of the pass's, so U = running list ++ pass, n = r + count entries;
//   2. radix select: six rounds of an 11-bit shared-memory histogram over the keys that match the digits fixed so
//      far find T, the kk-th largest key of U exactly (kk = min(k, n));
//   3. order-preserving compaction (cub::DeviceSelect): the positions with key > T (fewer than kk), then those with
//      key == T.  All of the first and the leading kk - |first| of the second are the kk best: the running list holds
//      lower indices than the pass and lists equal keys by index, the pass is in index order, so the leading equal
//      entries are the lowest-index ones however many millions tie;
//   4. a stable descending radix sort of those kk (key, index) pairs is the new running list: value descending,
//      ties by ascending index.
// Memory is O(k + pass), never O(m), and every step is deterministic.
#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "common.cuh"

namespace {

constexpr int RS_BITS = 11, RS_BINS = 1 << RS_BITS;   // one radix-select digit
constexpr int FIND_THREADS = RS_BINS / 2;             // k_topk_find: two bins per thread
constexpr int HIST_THREADS = 512;

struct SelState {
  unsigned long long prefix, mask;   // digits of T fixed so far (prefix == T after the last round)
  unsigned long long want;           // rank (1-based, from the top) of T among the keys that match prefix
  long long n_gt, n_eq;              // sizes of the two compactions
  unsigned int hist[RS_BINS];
};

__device__ __forceinline__ unsigned long long order_key(double v) {
  if (isnan(v)) v = -INFINITY;
  if (v == 0.0) v = 0.0;
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ double key_value(unsigned long long key) {
  return __longlong_as_double((long long)((key >> 63) ? (key & 0x7fffffffffffffffull) : ~key));
}

// U[0, r) = the running list's keys; U[r, r + count) holds the pass's values as doubles and becomes their keys in place
__global__ void k_topk_keys(unsigned long long *__restrict__ U, long long r, long long count,
                            const unsigned long long *__restrict__ run_keys, SelState *__restrict__ ss,
                            long long kk) {
  const long long n = r + count;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x)
    U[t] = t < r ? run_keys[t] : order_key(__longlong_as_double((long long)U[t]));
  if (blockIdx.x == 0) {
    for (int b = threadIdx.x; b < RS_BINS; b += blockDim.x) ss->hist[b] = 0;
    if (threadIdx.x == 0) { ss->prefix = ss->mask = 0; ss->want = (unsigned long long)kk; }
  }
}

__global__ void __launch_bounds__(HIST_THREADS) k_topk_hist(const unsigned long long *__restrict__ U, long long n,
                                                            SelState *__restrict__ ss, int shift) {
  __shared__ unsigned int sh[RS_BINS];
  for (int b = threadIdx.x; b < RS_BINS; b += blockDim.x) sh[b] = 0;
  __syncthreads();
  const unsigned long long prefix = ss->prefix, mask = ss->mask;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
    const unsigned long long key = U[t];
    if ((key & mask) == prefix) atomicAdd(&sh[(key >> shift) & (RS_BINS - 1)], 1u);
  }
  __syncthreads();
  for (int b = threadIdx.x; b < RS_BINS; b += blockDim.x)
    if (sh[b]) atomicAdd(&ss->hist[b], sh[b]);
}

// the bin that holds the want-th largest key: fixes the digit at `shift` (`bits` wide) and clears the histogram
__global__ void __launch_bounds__(FIND_THREADS) k_topk_find(SelState *__restrict__ ss, int shift, int bits) {
  using Scan = cub::BlockScan<unsigned int, FIND_THREADS>;
  __shared__ typename Scan::TempStorage tmp;
  const int b0 = RS_BINS - 1 - 2 * threadIdx.x, b1 = b0 - 1;    // bins in descending order
  const unsigned int c0 = ss->hist[b0], c1 = ss->hist[b1];
  const unsigned long long want = ss->want;
  unsigned int above;
  Scan(tmp).ExclusiveSum(c0 + c1, above);
  int digit = -1;
  unsigned long long rest = 0;
  if (above < want && want <= (unsigned long long)above + c0) { digit = b0; rest = want - above; }
  else if ((unsigned long long)above + c0 < want && want <= (unsigned long long)above + c0 + c1) {
    digit = b1; rest = want - above - c0;
  }
  if (digit >= 0) {
    ss->prefix |= (unsigned long long)digit << shift;
    ss->mask |= ((1ull << bits) - 1) << shift;
    ss->want = rest;
  }
  ss->hist[b0] = 0;
  ss->hist[b1] = 0;
}

struct KeyCmp {                     // compaction test of position i against T: key > T (gt) or key == T
  const unsigned long long *U;
  const SelState *ss;
  int gt;
  __device__ bool operator()(long long i) const {
    const unsigned long long key = U[i], T = ss->prefix;
    return gt ? key > T : key == T;
  }
};

// the kk selected entries in U order: every key > T, then the leading key == T ones
__global__ void k_topk_gather(const unsigned long long *__restrict__ U, long long r, long long base,
                              const long long *__restrict__ run_idx, const long long *__restrict__ gt_pos,
                              const long long *__restrict__ eq_pos, const SelState *__restrict__ ss, long long kk,
                              unsigned long long *__restrict__ keys_out, long long *__restrict__ idx_out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= kk) return;
  const long long g = ss->n_gt;
  const long long pos = t < g ? gt_pos[t] : eq_pos[t - g];
  keys_out[t] = U[pos];
  idx_out[t] = pos < r ? run_idx[pos] : base + (pos - r);
}

__global__ void k_topk_out(const unsigned long long *__restrict__ run_keys, const long long *__restrict__ run_idx,
                           long long kk, int k, ombo_best *__restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= k) return;
  out[t].value = t < kk ? key_value(run_keys[t]) : -INFINITY;
  out[t].index = t < kk ? run_idx[t] : -1;
}

}  // namespace

extern "C" int ombo_score_topk(ombo_ctx *ctx, const ombo_gp *gps, int n_gp, const ombo_pool *pool,
                               const ombo_acq *acq, int precision, int k, ombo_best *topk_dev, void *stream) {
  int rc = ombo_validate_score(ctx, gps, n_gp, pool, acq, precision);
  if (rc) return rc;
  OMBO_CHECK(acq->kind != OMBO_ACQ_NONE, "score_topk: needs an acquisition");
  OMBO_CHECK(k >= 1 && k <= OMBO_TOPK_MAX, "score_topk: k=%d out of range (1..%d)", k, OMBO_TOPK_MAX);
  OMBO_CHECK(topk_dev != nullptr, "score_topk: topk_dev is NULL");
  OMBO_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  const long long m = pool->m;
  const long long chunk = std::min(1LL << ctx->knobs.chunk_log2, std::max(m, 1LL));
  const long long n_max = k + chunk;

  // workspace: selection state | U | running list | sort input | > T positions | == T positions | cub scratch
  const cub::CountingInputIterator<long long> ids(0);
  size_t sel_bytes = 0, sort_bytes = 0;
  OMBO_CUDA(cub::DeviceSelect::If(nullptr, sel_bytes, ids, (long long *)nullptr, (long long *)nullptr, n_max,
                                  KeyCmp{nullptr, nullptr, 0}, s));
  OMBO_CUDA(cub::DeviceRadixSort::SortPairsDescending(nullptr, sort_bytes, (unsigned long long *)nullptr,
                                                      (unsigned long long *)nullptr, (long long *)nullptr,
                                                      (long long *)nullptr, k, 0, 64, s));
  auto up = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t o_U = up(sizeof(SelState)), o_run = o_U + up((size_t)n_max * 8), o_sort = o_run + up((size_t)k * 16),
               o_gt = o_sort + up((size_t)k * 16), o_eq = o_gt + up((size_t)k * 8),
               o_cub = o_eq + up((size_t)n_max * 8);
  rc = ombo_ws_reserve(&ctx->ws_topk, &ctx->ws_topk_bytes, o_cub + std::max(sel_bytes, sort_bytes));
  if (rc) return rc;
  char *ws = (char *)ctx->ws_topk;
  SelState *ss = (SelState *)ws;
  unsigned long long *U = (unsigned long long *)(ws + o_U);
  unsigned long long *run_keys = (unsigned long long *)(ws + o_run);
  long long *run_idx = (long long *)(run_keys + k);
  unsigned long long *sort_keys = (unsigned long long *)(ws + o_sort);
  long long *sort_idx = (long long *)(sort_keys + k);
  long long *gt_pos = (long long *)(ws + o_gt), *eq_pos = (long long *)(ws + o_eq);
  void *cub_tmp = ws + o_cub;

  const size_t esz = pool->dtype == 0 ? 8 : 4;
  const int hist_blocks = std::max(1, std::min((int)((n_max + HIST_THREADS - 1) / HIST_THREADS), 2 * ctx->num_sms));
  long long r = 0;                                          // entries of the running list
  for (long long first = 0; first < m; first += chunk) {
    const long long count = std::min(chunk, m - first);
    ombo_pool sub = *pool;
    sub.m = count;
    sub.index_base = pool->index_base + first;
    sub.X = pool->X ? (const char *)pool->X + (size_t)first * pool->d * esz : nullptr;
    rc = ombo_score_pass(ctx, gps, n_gp, &sub, sub.X, 0, count, acq, precision, nullptr, nullptr, (double *)(U + r),
                         count, nullptr, s);
    if (rc) return rc;
    const long long n = r + count, kk = std::min((long long)k, n);
    k_topk_keys<<<(unsigned)std::min((n + 255) / 256, 8LL * ctx->num_sms), 256, 0, s>>>(U, r, count, run_keys, ss,
                                                                                          kk);
    ctx->launches += 1;
    OMBO_CUDA(cudaGetLastError());
    for (int hi = 64; hi > 0; hi -= RS_BITS) {              // digits [53, 64), [42, 53), ..., [0, 9)
      const int lo = std::max(0, hi - RS_BITS);
      k_topk_hist<<<hist_blocks, HIST_THREADS, 0, s>>>(U, n, ss, lo);
      k_topk_find<<<1, FIND_THREADS, 0, s>>>(ss, lo, hi - lo);
      ctx->launches += 2;
      OMBO_CUDA(cudaGetLastError());
    }
    OMBO_CUDA(cub::DeviceSelect::If(cub_tmp, sel_bytes, ids, gt_pos, &ss->n_gt, n, KeyCmp{U, ss, 1}, s));
    OMBO_CUDA(cub::DeviceSelect::If(cub_tmp, sel_bytes, ids, eq_pos, &ss->n_eq, n, KeyCmp{U, ss, 0}, s));
    k_topk_gather<<<(unsigned)((kk + 255) / 256), 256, 0, s>>>(U, r, sub.index_base, run_idx, gt_pos, eq_pos, ss, kk,
                                                               sort_keys, sort_idx);
    ctx->launches += 3;
    OMBO_CUDA(cudaGetLastError());
    size_t sb = sort_bytes;
    // num_items as the same type (int) as in the size query: cub sizes its scratch per offset type
    OMBO_CUDA(cub::DeviceRadixSort::SortPairsDescending(cub_tmp, sb, sort_keys, run_keys, sort_idx, run_idx, (int)kk,
                                                        0, 64, s));
    ctx->launches += 1;
    r = kk;
  }
  k_topk_out<<<(unsigned)((k + 255) / 256), 256, 0, s>>>(run_keys, run_idx, r, k, topk_dev);
  ctx->launches += 1;
  OMBO_CUDA(cudaGetLastError());
  return OMBO_OK;
}
