// tcgen05 / TMA / mbarrier PTX wrappers and the parameter block shared by the fast-mode posterior kernels
// (posterior_fast.cu: 16-bit x3 planes, single CTA; posterior_fast8.cu: f8c planes, cta_group::2 pair).
#pragma once
#include <cuda.h>
#include <stdlib.h>

#include "candidates.cuh"

#define FM 128            // candidates per tile (UMMA M)
#define FK 64             // K-block: 64 bf16 = 128 B = one swizzle atom row
// generator warps GW (template): 8 (one per 16-byte operand chunk of the K-block, R = 4 rows per lane) or
// 16 (two row halves, R = 2 rows per lane: more warps per scheduler to overlap the FMA / MUFU / ALU phases)
#define PLANE_BYTES (FM * 128)          // 16 KB
#define STAGE_BYTES (2 * PLANE_BYTES)   // 32 KB

// ---- PTX wrappers ------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_n(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
#ifndef MBAR_SUSPEND_HINT
#define MBAR_SUSPEND_HINT 0     // 1: try_wait carries a suspend-time hint (the thread sleeps in hardware until the phase flips)
#endif
__device__ __forceinline__ uint32_t mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t ok;
#if MBAR_SUSPEND_HINT
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(0x989680u)
      : "memory");
#else
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
#endif
  return ok;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try(bar, parity)) {}
}
// polling warps steal issue slots from the K1 generators: back off between probes
__device__ __forceinline__ void mbar_wait_sleep(uint32_t bar, uint32_t parity, unsigned ns) {
#if MBAR_SUSPEND_HINT
  while (!mbar_try(bar, parity)) {}
#else
  while (!mbar_try(bar, parity)) __nanosleep(ns);
#endif
}
// one lane of a CONVERGED warp; unlike `lane == 0` the compiler knows a single thread is active, so
// tcgen05 / TMA operands stay in uniform registers without a per-instruction waterfall loop
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "elect.sync _|P1, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, P1;\n"
      "}\n"
      : "=r"(pred));
  return pred;
}
#ifndef MMA_SLEEP_NS
#define MMA_SLEEP_NS 32    // back-off of the MMA issuer's barrier probes (0 = pure spin; measured equal)
#endif
__device__ __forceinline__ void mbar_wait_prof(uint32_t bar, uint32_t parity, unsigned ns, long long &acc, bool on) {
  if (!on) { if (ns) mbar_wait_sleep(bar, parity, ns); else mbar_wait(bar, parity); return; }
  long long t0 = clock64();
  mbar_wait_sleep(bar, parity, ns);
  acc += clock64() - t0;
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
// linear bulk copies (TMA without a tensor map): smem -> global with bulk-group completion,
// global -> smem with mbarrier transaction completion
__device__ __forceinline__ void bulk_store(void *gdst, uint32_t ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gdst), "r"(ssrc), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t sdst, const void *gsrc, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(sdst),
               "l"(gsrc), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t local, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(local), "r"(rank));
  return r;
}
// arrive / expect_tx on a barrier that may live in the peer CTA of the cluster, WITHOUT cluster-scope release semantics
// (default .release.cta, as CUTLASS' ClusterBarrier::arrive does): .release.cluster compiles to MEMBAR.ALL.GPU + ERRBAR, ~1000 cycles per
// arrive on the critical path of every generator warp (ncu source view, profiles/r02_*).  The data these arrivals
// publish sits in the arriving CTA's OWN shared memory, is ordered by the preceding fence.proxy.async / tcgen05 fence
// and is read through the async proxy after the barrier has completed -- shared memory has no cache to flush.
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_n_remote(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_remote(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(count) : "memory");
}
// 2-SM TMA load: data lands in this CTA's smem, the transaction bytes are counted on the LEADER's barrier
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap *map, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::"r"(dst),
      "l"(map), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {     // arrives on `bar` in BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t *v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// UMMA shared-memory descriptor, K-major, SWIZZLE_128B: rows of 128 B, 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t make_sdesc(uint32_t saddr) {
  const uint32_t lo = ((saddr & 0x3FFFF) >> 4) | (1u << 16);           // start address, LBO = 1 (unused)
  const uint32_t hi = 64u | (1u << 14) | (2u << 29);                   // SBO = 1024 B, version 1, SWIZZLE_128B
  return ((uint64_t)hi << 32) | lo;
}
// instruction descriptor: D = f32, A = B = bf16, both K-major, N = 128, M = 128

struct FastParams {
  GpDev gp;
  PoolDev pool;
  long long m;
  double *mu_out, *var_out;
  unsigned char *kcache;   // per-CTA cache of generated K* blocks (n_pad/64 x 32 KB), L2 resident
  long long *prof;   // optional per-CTA wait-cycle counters (timing experiments)
  int dbg;   // f8c kernel, OMBO_FAST_DBG: timing experiments (posterior_fast8.cu; results are garbage)
  const unsigned int *sched;   // f8c kernel: step schedule of one tile (posterior_fast8.cu)
  int n_steps;
  int sched_in_smem;           // set by the launcher when the table fits beside the operand rings
  long long *trace;  // optional event trace of CTA 0 (OMBO_FAST_PROFILE=2): [8 roles][F8_TRACE_N] of (clock << 8 | code)
  FuseAcq fuse;      // f8c kernel only
};


extern __shared__ __align__(1024) unsigned char fast_smem[];

// host helpers shared by the fast-mode translation units (posterior_fast.cu)
typedef CUresult (*PFN_encodeTiled_t)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                      const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled_t ombo_get_encode_tiled();
int ombo_make_linear_map(CUtensorMap *map, const void *base, size_t rows);
