// dmip_ptx.cuh — thin inline-PTX wrappers for the sm_100a features the kernels use:
// mbarrier, bulk-TMA (cp.async.bulk), tcgen05 (alloc / mma / commit / ld / st / fences) and the
// UMMA shared-memory + instruction descriptors.  No CUTLASS dependency.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dmip {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// One lane of a CONVERGED warp.  The single-thread instructions (tcgen05.mma / commit, bulk copies) are wrapped in
// `if (elect_one())` while the surrounding loop is executed by the whole warp: operands then stay provably
// warp-uniform and live in uniform registers.  (Issuing from inside an `if (lane == 0)` region instead makes ptxas
// emit an ELECT / R2UR.BROADCAST / BRA.U.ANY "waterfall" loop around every UTCHMMA — measured 5x slower issue.)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------ watchdog
// A dead-locked mbarrier wait would hang the GPU until the process is killed.  Every wait therefore
// carries a clock64() watchdog: after ~4e9 cycles it records (tag, block) and traps, which surfaces
// as cudaErrorLaunchFailure on the host instead of a hang.
static __device__ unsigned int g_watchdog_info[4];

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, uint32_t tag) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      g_watchdog_info[0] = 0xDEAD0000u | tag;
      g_watchdog_info[1] = blockIdx.x;
      g_watchdog_info[2] = threadIdx.x;
      g_watchdog_info[3] = parity;
      __threadfence_system();
      __trap();
    }
  }
}

// ------------------------------------------------------------------ async-proxy fence, bulk TMA
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// same copy, delivered to the same CTA-relative offset (data and mbarrier) of every CTA in `cta_mask`
__device__ __forceinline__ void bulk_g2s_multicast(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar,
                                                   uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::
          "r"(smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "h"(cta_mask)
      : "memory");
}

// ------------------------------------------------------------------ thread-block cluster
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {  // every thread of every CTA in the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ------------------------------------------------------------------ tensor memory
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_holder) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {  // same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// all previously issued tcgen05.mma of this thread arrive (once) on `bar` when they complete
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// the same arrival delivered to the barrier at this CTA-relative offset in every CTA of `cta_mask`
__device__ __forceinline__ void tc_commit_multicast(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}

// ------------------------------------------------------------------ CTA pair (cta_group::2)
// Two CTAs of a cluster (ranks 2i, 2i+1 — same TPC) run ONE tcgen05.mma of M = 256: each CTA owns 128 rows of A and D
// (its own shared / tensor memory, same CTA-relative addresses in both) and HALF of B (N/2 rows of the N x K tile in
// its own shared memory).  Only the even-rank ("leader") CTA issues mma / commit; alloc / dealloc are executed by one
// warp in EACH CTA.
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_holder) {  // one full warp in each CTA, same holder offset
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void umma_ss_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_ts_pair(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of all earlier pair-MMAs of this thread -> one arrival on the barrier at this CTA-relative offset in
// every CTA of `cta_mask`
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}
// address of `p` (a shared::cta address of THIS CTA) in the shared window of cluster CTA `rank`
__device__ __forceinline__ uint32_t mapa_u32(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
// arrive (release, cluster scope) on an mbarrier of another CTA of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}

// 16-byte store into the shared window of any CTA of the cluster (address from mapa_u32, or an own shared::cta address)
__device__ __forceinline__ void st_cluster_v4(uint32_t cluster_addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(cluster_addr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}
// asynchronous 16-byte store into ANOTHER CTA's shared memory; its completion is counted (16 bytes) on an mbarrier of that
// same CTA — the writer neither fences nor arrives (both addresses from mapa_u32 with the destination's rank)
__device__ __forceinline__ void st_async_v4(uint32_t cluster_addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d,
                                            uint32_t cluster_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(
                   cluster_addr),
               "r"(a), "r"(b), "r"(c), "r"(d), "r"(cluster_mbar)
               : "memory");
}
// generic-proxy writes into ANY CTA's shared memory of the cluster -> visible to the async proxy (tensor core operands)
__device__ __forceinline__ void fence_proxy_async_cluster_smem() {
  asm volatile("fence.proxy.async.shared::cluster;" ::: "memory");
}
// wait on an own mbarrier whose arrivals come from another CTA (release.cluster): acquire at cluster scope.
// (Every successful wait then invalidates L1 — CCTL.IVALL, 6 % of the forward loss kernel's warp samples.  With
// -DDMIP_CTA_ACQUIRE the acquire stays at CTA scope, as in CUTLASS' ClusterBarrier::wait — sufficient for waiters that
// only issue tcgen05.mma on async-proxy data afterwards; measured: no change of the step time (3.89 / 3.88 ms PINN,
// 1.171 / 1.183 ms DSM), so the formally stronger form stays.)
#ifdef DMIP_CTA_ACQUIRE
#define DMIP_TRY_WAIT_CLUSTER "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
#else
#define DMIP_TRY_WAIT_CLUSTER "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
#endif
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      DMIP_TRY_WAIT_CLUSTER
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity, uint32_t tag) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait_cluster(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      g_watchdog_info[0] = 0xDEAD0000u | tag;
      g_watchdog_info[1] = blockIdx.x;
      g_watchdog_info[2] = threadIdx.x;
      g_watchdog_info[3] = parity;
      __threadfence_system();
      __trap();
    }
  }
}

// the same arrival without release semantics: for a thread that publishes nothing of its own (relay of a TMA completion),
// or right after a fence that already ordered its stores (fence.proxy.async.shared::cluster carries a GPU-scope membar)
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}

// ------------------------------------------------------------------ descriptors
// Shared-memory operand descriptor, K-major, 128-byte swizzle, bf16:
//   rows (M or N index) are 128 B apart inside an 8-row / 1024 B swizzle atom, atoms are SBO = 1024 B apart,
//   16-byte chunk c of row r sits at chunk position c ^ (r & 7).  One descriptor covers one UMMA_K = 16
//   slice (32 B); advancing K inside the 64-element swizzle row adds 32 B to the start address.
//   bits [0,14) addr>>4 | [16,30) LBO>>4 (=1, unused for swizzled K-major) | [32,46) SBO>>4 | [46,48) version=1
//   | [61,64) layout type (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t umma_smem_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor (upper 32 bits of the 64-bit idesc), kind::f16, A/B = bf16 K-major, D = fp32.
//   [4,6) D fmt (1 = f32) | [7,10) A fmt (1 = bf16) | [10,13) B fmt (1 = bf16) | 15 A major (0 = K) |
//   16 B major (0 = K) | [17,23) N>>3 | [24,29) M>>4
__host__ __device__ constexpr uint32_t umma_idesc_bf16(uint32_t M, uint32_t N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
// same with A = B = f16 (format 0).  Mixing f16 activations with bf16 weights in one instruction traps on B200.
__host__ __device__ constexpr uint32_t umma_idesc_f16(uint32_t M, uint32_t N) {
  return (1u << 4) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// General form of the two above: operand formats bf16, D = fp32; a_mn / b_mn = 1 selects the MN-major ("transposed")
// shared-memory layout of that operand (bit 15 / bit 16).
__host__ __device__ constexpr uint32_t umma_idesc_bf16_major(uint32_t M, uint32_t N, uint32_t a_mn, uint32_t b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (a_mn << 15) | (b_mn << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
// Shared-memory operand descriptor, 128-byte swizzle, with explicit leading / stride byte offsets.
//   K-major : rows of 64 k (128 B); 8 rows = one 1024 B atom; SBO = distance between 8-row groups; LBO unused (16 B).
//   MN-major: lines of 64 MN elements (128 B); 8 consecutive k = one 1024 B atom; LBO = distance between 64-element
//             MN groups, SBO = distance between 8-k groups (CUTLASS canonical ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16 B units).
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Byte offset of element (mn, k) of an MN-major SWIZZLE_128B bf16 image (see umma_smem_desc): the 16-byte chunk
// holding MN elements 8c .. 8c+7 of line k sits at chunk position c ^ (k & 7).
__host__ __device__ __forceinline__ uint32_t mn128_offset(uint32_t mn, uint32_t k, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  const uint32_t line = k & 7u, c = (mn & 63u) >> 3;
  return (mn >> 6) * lbo_bytes + (k >> 3) * sbo_bytes + line * 128u + ((c ^ line) << 4) + (mn & 7u) * 2u;
}

// D[tmem] (+)= A[smem] * B[smem]^T      (issued by ONE thread)
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T      (A: lane = row, 32-bit column c holds k = 2c (low half), 2c+1 (high half))
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ------------------------------------------------------------------ TMEM <-> registers (32 lanes x 32 bit, xN columns)
// Warp w of a CTA may touch TMEM lanes [32*(w%4), 32*(w%4)+32); thread i of the warp gets lane 32*(w%4)+i.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void red_add_f32(float* gptr, float v) {   // fire-and-forget fp32 atomic add (SASS: RED)
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(gptr), "f"(v) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// ------------------------------------------------------------------ math helpers
__device__ __forceinline__ float tanh_fast(float x) {  // MUFU.TANH, max rel. error 2^-11
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// tanh(u) for |u| <= 1 (u is itself a tanh): odd minimax polynomial u (c0 + c1 s + c2 s^2 + c3 s^3), s = u^2, max abs
// error 3.3e-5 — 1/60 of the bf16 half-ulp the result is rounded to — in 5 FMA-pipe operations, so the second tanh of
// layer 0 (SURVEY.md Q1) runs beside the MUFU instead of on it.
__device__ __forceinline__ float tanh_unit_poly(float u) {
  const float t = u * u;
  float p = -0.024654336273670197f;
  p = fmaf(p, t, 0.1154140904545784f);
  p = fmaf(p, t, -0.3288920521736145f);
  p = fmaf(p, t, 0.999693751335144f);
  return u * p;
}
// ---- packed fp32x2 arithmetic (sm_100: FADD2 / FMUL2 / FFMA2).  Each lane is the same IEEE round-to-nearest operation as
// the scalar `+` / `*` / fmaf, so a packed rewrite that keeps the operation order keeps every result bit.
__device__ __forceinline__ unsigned long long f32x2_pack(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f32x2_unpack(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long f32x2_add(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ unsigned long long f32x2_mul(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ unsigned long long f32x2_fma(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
// tanh_unit_poly on a packed pair: same coefficients, same operation order, bit-identical per lane
__device__ __forceinline__ unsigned long long tanh_unit_poly_f32x2(unsigned long long u) {
  const unsigned long long t = f32x2_mul(u, u);
  unsigned long long p = f32x2_fma(f32x2_pack(-0.024654336273670197f, -0.024654336273670197f), t,
                                   f32x2_pack(0.1154140904545784f, 0.1154140904545784f));
  p = f32x2_fma(p, t, f32x2_pack(-0.3288920521736145f, -0.3288920521736145f));
  p = f32x2_fma(p, t, f32x2_pack(0.999693751335144f, 0.999693751335144f));
  return f32x2_mul(u, p);
}
// ---- packed f16x2 epilogue math: the hidden activations are tanh values in (-1, 1), where f16 carries 11 mantissa
// bits against bf16's 8, and every instruction below handles two elements (half the issue slots of the f32 versions)
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {   // element with the lower index in bits [0,16)
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// the same with saturation to +-65504 (one F2FP.SATFINITE): round-then-saturate equals clamp-then-round for every non-NaN
// input because 65504 is the largest finite f16; a NaN stays NaN
__device__ __forceinline__ uint32_t pack_f16x2_sat(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t tanh_f16x2(uint32_t x) {           // MUFU.TANH.F16x2
  uint32_t y;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}
__device__ __forceinline__ uint32_t hmul2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("mul.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t hfma2(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
// tanh_unit_poly on a packed pair, coefficients rounded to f16: max abs error 5.9e-4 over |u| <= tanh(1)... (the bf16
// rounding this replaces had 2.0e-3)
__device__ __forceinline__ uint32_t tanh_unit_poly_f16x2(uint32_t u) {
  const uint32_t t = hmul2(u, u);
  uint32_t p = hfma2(0xa650a650u, t, 0x2f632f63u);   // -0.024658, 0.115417
  p = hfma2(p, t, 0xb543b543u);                      // -0.328857
  p = hfma2(p, t, 0x3bff3bffu);                      //  0.999512
  return hmul2(u, p);
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {  // element with the lower index in bits [0,16)
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float bf16_round(float x) {  // value of x after rounding to bf16
  return __uint_as_float(pack_bf16x2(x, 0.f) << 16);
}

// Byte offset of element (row, k) inside a K-major SWIZZLE_128B bf16 tile whose K-blocks (64 elements) are
// `kblock_bytes` apart (= rows * 128).  Used by every producer of an operand image (pack kernel, A0 builder,
// epilogue) so that they agree with umma_smem_desc_sw128 by construction.
__host__ __device__ __forceinline__ uint32_t sw128_offset(uint32_t row, uint32_t k, uint32_t kblock_bytes) {
  const uint32_t kb = k >> 6, kin = k & 63u;
  const uint32_t chunk = (kin >> 3) ^ (row & 7u);
  return kb * kblock_bytes + (row >> 3) * 1024u + (row & 7u) * 128u + chunk * 16u + (kin & 7u) * 2u;
}

}  // namespace dmip
