// dmip_tc.cu — the tcgen05 path: persistent fused Euler–Maruyama sampler (K1) and score-net forward.
//
// One CTA per SM, 128 particles (rows) per tile, the whole S-step reverse SDE of a tile runs on chip.  20 warps:
//
//   warps 0-15    ROW warps, four threads per particle row (warp w: TMEM lane quarter w % 4, column group w / 4).
//                 Hidden layers: tcgen05.ld accumulator -> +bias -> tanh (twice after layer 0, SURVEY.md Q1) -> bf16 ->
//                 next layer's A operand (tcgen05.st, or swizzled st.shared); 4 warps per scheduler keep the MUFU pipe
//                 (the epilogue's bound: one tanh per activation) busy while the tensor pipe runs the next chunk.
//                 State: each thread keeps its share of the particle's fp32 SDE state in REGISTERS for the whole
//                 integration, draws the Philox noise and applies the drift/diffusion update in the shadow of the
//                 MMA-bound layers, reads the output layer's accumulator and builds the next step's layer-0 operand
//                 (bf16 hi/lo split).  y and t never enter the GEMM: they are constant over a tile and are folded,
//                 in fp32, into a per-step layer-0 bias  b0 + W0[:,y]·y + tau·W0[:,t].
//   warp 16       bulk-TMA producer: streams the net's bf16 weight stages (16 KB = 128 out-features x 64 k, K-major,
//                 128B-swizzled — written in exactly that image by dmip_pack.cu) from L2 into a 5-deep shared-memory
//                 ring, the same ~1.3 MB sequence every step; the two CTAs of a cluster each fetch half of every stage
//                 and multicast it to both.
//   warp 17       MMA issuer (one elected lane): per layer four N=128 accumulator chunks of
//                 tcgen05.mma.cta_group::1.kind::f16 (bf16 x bf16 -> fp32 in TMEM).  The activations are the A operand
//                 and ALTERNATE between shared memory and tensor memory from layer to layer
//                 (A0: smem -> H1: tmem -> H2: smem -> H3: tmem), so an epilogue never overwrites the operand its own
//                 layer's MMAs still read, and the epilogue of chunk c overlaps the MMAs of chunk c+1.
//                 Producer and issuer sit at the HIGHEST warp ids: the warp scheduler prefers high ids, and an issuer
//                 at warp 1 was measured starved by the math warps (200 instead of 75 cycles per MMA).
//   warps 18-19   idle: registers are allocated in units of four warps, so they exist anyway; setmaxnreg hands the
//                 spare registers of warps 16-19 to the row warps.
//
// Reference code replaced: models/diffusion.py:27-46,158-180; sdes.py:21-49,77-87; nets.py:17-57,143-157.
#include <stdlib.h>

#include "dmip_common.h"
#include "dmip_ptx.cuh"
#include "dmip_rng.cuh"
#include "dmip_sde.cuh"

namespace dmip {

namespace {

constexpr int kTileM = 128;
constexpr int kStageBytes = 16384;   // 128 rows x 64 k x bf16: one K-block of a 128-feature chunk
constexpr int kNumSlots = 6;         // ring of 16 KB slots, filled / waited for / released in PAIRS (32 KB = 8 MMAs):
constexpr int kNumPairs = kNumSlots / 2;   // a barrier wait costs ~85 cycles in the issuing thread and the tensor core
constexpr int kPairBytes = 2 * kStageBytes;  // queues only ~1 MMA ahead, so waits per MMA decide the MMA rate
constexpr int kHBytes = 131072;      // 128 rows x 512 k x bf16 = 8 K-blocks
constexpr int kThreads = 640;        // warps: 0-15 row warps (epilogue + state), 16 producer, 17 MMA, 18-19 idle
constexpr int kRegsSmall = 32;       // registers are allocated per 4 warps (18 warps are billed as 20), so the kernel
constexpr int kRegsRow = 112;        // launches with 640 x 96 and setmaxnreg moves 128 x 64 of them to the row warps
constexpr int kNumRowWarps = 16;
constexpr int kRowThreads = 512;
constexpr int kProducerWarp = 16;
constexpr int kMmaWarp = 17;
#ifndef DMIP_CLUSTER
#define DMIP_CLUSTER 2
#endif
constexpr int kCluster = DMIP_CLUSTER;   // CTAs per cluster sharing one multicast weight stream (2; 4 is a build-time experiment)
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kTmemH = 0;       // 256 columns: 128 x 512 bf16 activations (A operand)
constexpr uint32_t kTmemAcc = 256;   // 2 x 128 columns: fp32 accumulator chunks
// l0_split = 4, CDE / DPS samplers: the f16 layer-0 operand (<= 128 k = 64 columns) sits in the LAST quarter of the
// activation columns.  H1 / H3 chunk 3 overwrites them only after the layer's last MMA has retired, chunks 0-2 never touch
// them, and the output layer (which reads all of H3) is complete before the next operand is written — so layer 0 runs
// tensor-memory A operands (0.5 N + 13 cycles per instruction instead of 0.5 N + 46).
constexpr uint32_t kTmemL0 = kTmemH + 192;
// The same quarter serves layer 2: the epilogue of layer 1's LAST chunk (features 384-511 of H2 = layer 2's K-blocks 6, 7)
// starts after every MMA of layer 1 has retired, so H1 is dead and that chunk can land in columns 192-255 instead of
// shared memory; H3's chunk 3 replaces it only after layer 2's last MMA.  A quarter of layer 2's instructions then read a
// tensor-memory A operand (0.5 N + 13 cycles instead of 0.5 N + 46).  -DDMIP_L2_TAIL_TMEM=0 restores all-shared H2.
#ifndef DMIP_L2_TAIL_TMEM
#define DMIP_L2_TAIL_TMEM 1
#endif
constexpr bool kL2TailTmem = DMIP_L2_TAIL_TMEM != 0;

// shared-memory map (offsets from the 1024-aligned dynamic shared memory base; 231.6 of the 232.4 KB a CTA may have)
constexpr int kOffH = 0;
constexpr int kOffB = kOffH + kHBytes;
constexpr int kOffB0 = kOffB + kNumSlots * kStageBytes;   // float[512] effective layer-0 bias of the coming pass
constexpr int kOffB3 = kOffB0 + 2048;                     // float[128] output-layer bias (DPS: [0,8) prior net, [8,16) likelihood net)
constexpr int kOffBar = kOffB3 + 512;
constexpr int kNumBars = 2 * kNumPairs + 2 + 2 + 1 + 1 + 1 + 4 + 1;
constexpr int kOffTmem = kOffBar + kNumBars * 8;
constexpr int kSmemBytes = kOffTmem + 16;

enum { kModeSampler = 0, kModeForward = 1 };

struct TcNetDev {
  const uint8_t* stages;
  const float* b0;
  const float* b1;
  const float* b2;
  const float* b3;
  const float* w0c;  // [512][n_const]
  int kb0, ksteps0, dv, split, l0_f16, outpad, n_const, n_stages;
  int l0_tmem;   // the (single f16 part) layer-0 operand lives in tensor memory, columns kTmemL0 .. (TS MMAs instead of SS);
                 // host-side only: selects the k_tc_mlp<.., .., L0TMEM> instantiation
};

struct TcParams {
  int mode, variant, n_nets;
  TcNetDev net[2];
  int xdim, ydim, n_obs, tiles_per_obs, S;
  long long n_per_obs, n_tiles;
  float T, bmin, bmax, mean, std, delta, sqrt_delta;   // bmin / bmax: beta range (VP) or sigma range (VE)
  int sde_kind, n_corr;     // dmip_sde.cuh: forward SDE and corrector sub-steps per step
  float snr;
  const float* y;
  float* out;
  int rng_mode;
  unsigned long long seed, gidx_base;
  const float* x0;
  const float* noise;
  const float* ynoise;
  // forward mode
  const float* fx;
  const float* fcond;
  const float* ft;
  int fx_dim, fcond_dim, out_dim;
  int dbg;                  // debug bits (DMIP_DBG): 1 = no weight copies, 2 = no MMA issue, 4 = 3-deep ring
  int cluster;              // CTAs per cluster sharing one multicast weight stream (1, 2 or 4)
  unsigned long long* tl;   // optional timeline buffer (debug): 4 role segments of [count, (clock << 16 | code)...]
  int tl_cap;
};

struct Bars {
  uint64_t* full;       // [kNumPairs]   weight slot pair landed        (tx bytes)
  uint64_t* empty;      // [kNumPairs]   weight slot pair consumed      (one tcgen05.commit per cluster CTA)
  uint64_t* acc_full;   // [2]           hidden accumulator chunk complete  (tcgen05.commit)
  uint64_t* acc_empty;  // [2]           hidden chunk drained               (16 row warps)
  uint64_t* out_full;   // [1]           output-layer chunk complete        (tcgen05.commit)
  uint64_t* out_empty;  // [1]           output-layer chunk drained         (16 row warps)
  uint64_t* sh_free;    // [1]           layer 2 has consumed the shared-memory operand region (tcgen05.commit)
  uint64_t* hready;     // [4]           K-blocks 2c, 2c+1 of the next A operand written (16 row warps)
  uint64_t* a0_ready;   // [1]           layer-0 operand + bias of the next pass written (16 row warps)
};

// Kernel parameters live in the constant bank; ptxas re-materialises them with an LDC at every use after an asm with a
// "memory" clobber (all mbarrier / tcgen05 / TMA wrappers) — ~40 cycles each in the producer's and the issuer's
// dependent chains.  A value that went through a warp shuffle cannot be re-materialised and stays in a register.
// (All lanes hold the same parameter value, so the shuffle is the identity.)
__device__ __forceinline__ int keep(int v) { return __shfl_sync(0xffffffffu, v, 0); }
__device__ __forceinline__ long long keep(long long v) {
  const unsigned lo = __shfl_sync(0xffffffffu, static_cast<unsigned>(v), 0);
  const unsigned hi = __shfl_sync(0xffffffffu, static_cast<unsigned>(static_cast<unsigned long long>(v) >> 32), 0);
  return static_cast<long long>((static_cast<unsigned long long>(hi) << 32) | lo);
}
template <class T>
__device__ __forceinline__ const T* keep(const T* p) {
  return reinterpret_cast<const T*>(keep(static_cast<long long>(reinterpret_cast<uintptr_t>(p))));
}

// identity the compiler cannot see through or move: ties a computation to this point of the instruction stream
__device__ __forceinline__ uint32_t pin_here(uint32_t v) {
  asm volatile("" : "+r"(v) :: "memory");
  return v;
}

template <int kRegs>
__device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegs)); }
template <int kRegs>
__device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegs)); }

__device__ __forceinline__ void st_shared_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(smem_u32(p)), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// ------------------------------------------------------------------------------------------------ hidden-layer epilogue
// One thread: row `row` (TMEM lane), 32 of the 128 columns of accumulator chunk `chunk` (column group `cgp`), as two
// 16-column halves so that the second half's tcgen05.ld is in flight while the first half's tanh runs.
// Build-time experiment -DDMIP_H_F16 (csrc/build.sh DMIP_DEFS): hidden activations and the weights of layers 1-3 in
// f16 instead of bf16 (kind::f16 traps when the two operand formats differ).  Measured on B200, synthetic config:
// errors vs the fp32 oracle halve (forward 7.2e-4 -> 2.3e-4 ... 3.7e-4, sampler cases 1.5-2x), but the power-capped
// clock drops and throughput falls 2-3 % (7.80e8 -> 7.55e8 ... 7.66e8 evals/s) with every epilogue variant below
// (DMIP_EPI 0: packed MUFU.TANH.F16x2 + HFMA2 polynomial, 1: fp32 math + f16 pack, 2: fp32 MUFU + packed polynomial),
// so bf16 stays the default.
#ifndef DMIP_EPI
#define DMIP_EPI 1
#endif
// 16 bytes of shared memory (shared-window address): LDS.128, where a generic pointer costs an LD.E.128.  Volatile with a
// memory clobber: the effective layer-0 bias is rewritten between passes, so the load must stay inside its pass.
__device__ __forceinline__ float4 ld_shared_v4f(uint32_t addr) {
  float4 r;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr) : "memory");
  return r;
}

template <bool kDoubleTanh>
__device__ __forceinline__ void tanh_pack16(const uint32_t (&v)[16], const float* __restrict__ bias, uint32_t (&pk)[8]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    // layer 0 (double tanh): the per-step effective bias in shared memory; layers 1-2: global, read-only path
    const float4 bq = kDoubleTanh ? ld_shared_v4f(smem_u32(bias + q * 4))
                                  : __ldg(reinterpret_cast<const float4*>(bias + q * 4));
#ifndef DMIP_H_F16
    // Packed pairs: bias add (FADD2) and the second tanh (Q1) as FMUL2 + 3 FFMA2 + FMUL2 on the FMA pipe, which the MUFU
    // (one scalar MUFU.TANH per activation, the epilogue's bound) leaves idle.  Lane-wise identical to the scalar forms.
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const unsigned long long z = f32x2_add(f32x2_pack(__uint_as_float(v[q * 4 + 2 * h]), __uint_as_float(v[q * 4 + 2 * h + 1])),
                                             h == 0 ? f32x2_pack(bq.x, bq.y) : f32x2_pack(bq.z, bq.w));
      float z0, z1;
      f32x2_unpack(z, z0, z1);
      unsigned long long t = f32x2_pack(tanh_fast(z0), tanh_fast(z1));
      if (kDoubleTanh) t = tanh_unit_poly_f32x2(t);
      float a0, a1;
      f32x2_unpack(t, a0, a1);
      pk[q * 2 + h] = pack_bf16x2(a0, a1);
    }
#else
    // hidden activations are f16 (tanh values in (-1, 1): 11 mantissa bits against bf16's 8; layers 1-3 weights are f16 too)
#if DMIP_EPI == 0      // everything packed: one MUFU.TANH.F16x2 per pair, second tanh (Q1) as an HFMA2 polynomial
    uint32_t t01 = tanh_f16x2(pack_f16x2(__uint_as_float(v[q * 4 + 0]) + bq.x, __uint_as_float(v[q * 4 + 1]) + bq.y));
    uint32_t t23 = tanh_f16x2(pack_f16x2(__uint_as_float(v[q * 4 + 2]) + bq.z, __uint_as_float(v[q * 4 + 3]) + bq.w));
    if (kDoubleTanh) {
      t01 = tanh_unit_poly_f16x2(t01);
      t23 = tanh_unit_poly_f16x2(t23);
    }
#elif DMIP_EPI == 1    // fp32 math, f16 only as the storage format
    float a[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float bb = e == 0 ? bq.x : e == 1 ? bq.y : e == 2 ? bq.z : bq.w;
      float t = tanh_fast(__uint_as_float(v[q * 4 + e]) + bb);
      if (kDoubleTanh) t = tanh_unit_poly(t);
      a[e] = t;
    }
    uint32_t t01 = pack_f16x2(a[0], a[1]), t23 = pack_f16x2(a[2], a[3]);
#else                  // fp32 MUFU, packed polynomial
    float a[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float bb = e == 0 ? bq.x : e == 1 ? bq.y : e == 2 ? bq.z : bq.w;
      a[e] = tanh_fast(__uint_as_float(v[q * 4 + e]) + bb);
    }
    uint32_t t01 = pack_f16x2(a[0], a[1]), t23 = pack_f16x2(a[2], a[3]);
    if (kDoubleTanh) {
      t01 = tanh_unit_poly_f16x2(t01);
      t23 = tanh_unit_poly_f16x2(t23);
    }
#endif
    pk[q * 2] = t01;
    pk[q * 2 + 1] = t23;
#endif
  }
}

struct NoExtra {
  __device__ __forceinline__ void operator()() const {}
};

// `extra` runs between the accumulator read and the tanh math, in the same straight-line block: independent ALU work
// placed there (the Philox draw of the state pre-update) is interleaved by the scheduler with the MUFU-bound tanh
// sequence instead of running after it.
template <bool kDoubleTanh, bool kToTmem, class Extra = NoExtra>
__device__ __forceinline__ void epi_hidden(uint32_t lane_taddr, uint32_t acc_col, int cgp, int row, int chunk, int lane,
                                           const float* __restrict__ bias, uint8_t* sH, uint64_t* acc_empty,
                                           uint64_t* hready, Extra extra = NoExtra()) {
  // Two 16-column halves, one in registers at a time (the particle state and the noise draw live in registers too):
  // the accumulator buffer is released after the second half's load — the issuer needs it two chunks later.
  const int n0 = chunk * 128 + cgp * 32;
  uint32_t v[16], pk[8];
  tmem_ld16(lane_taddr + acc_col + cgp * 32, v);
  tc_wait_ld();
  extra();
  tanh_pack16<kDoubleTanh>(v, bias + n0, pk);
  uint8_t* rowp = sH + (chunk * 2 + (cgp >> 1)) * kStageBytes + (row >> 3) * 1024 + (row & 7) * 128;
  const int c0 = (cgp & 1) * 4;   // K index n0 .. n0+31 -> K-block chunk*2 + (cgp>>1), 16-byte chunks c0 .. c0+3
  if (kToTmem) {
    tmem_st8(lane_taddr + kTmemH + static_cast<uint32_t>(n0 >> 1), pk);
  } else {
    st_shared_v4(rowp + (((c0 + 0) ^ (row & 7)) << 4), pk[0], pk[1], pk[2], pk[3]);
    st_shared_v4(rowp + (((c0 + 1) ^ (row & 7)) << 4), pk[4], pk[5], pk[6], pk[7]);
  }
  tmem_ld16(lane_taddr + acc_col + cgp * 32 + 16, v);
  tc_wait_ld();
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive(acc_empty);  // this warp's part of the chunk is in registers: the buffer may be reused
  tanh_pack16<kDoubleTanh>(v, bias + n0 + 16, pk);
  if (kToTmem) {
    tmem_st8(lane_taddr + kTmemH + static_cast<uint32_t>(n0 >> 1) + 8, pk);
    tc_wait_st();
    tc_fence_before();
  } else {
    st_shared_v4(rowp + (((c0 + 2) ^ (row & 7)) << 4), pk[0], pk[1], pk[2], pk[3]);
    st_shared_v4(rowp + (((c0 + 3) ^ (row & 7)) << 4), pk[4], pk[5], pk[6], pk[7]);
    fence_proxy_async_smem();
  }
  __syncwarp();
  if (lane == 0) mbar_arrive(hready);
}

// write one bf16 element of the layer-0 operand tile
__device__ __forceinline__ void a0_store(uint8_t* sH, int row, int k, float v) {
  const uint32_t off = sw128_offset(static_cast<uint32_t>(row), static_cast<uint32_t>(k), kStageBytes);
  const unsigned short h = static_cast<unsigned short>(pack_bf16x2(v, 0.f) & 0xFFFFu);
  *reinterpret_cast<unsigned short*>(sH + off) = h;
}
// l0_split = 4: the layer-0 operand is ONE f16 part (11 mantissa bits; |x| saturated to the f16 range) — the MMA count of
// plain bf16 with 8x its resolution of the state.  A NaN state element enters the net as NaN (a clamp would have fed it
// -65504): only that particle's own row sees it, and its fp32 state is NaN either way, so no sample changes.
__device__ __forceinline__ void a0_store_f16(uint8_t* sH, int row, int k, float v) {
  const uint32_t off = sw128_offset(static_cast<uint32_t>(row), static_cast<uint32_t>(k), kStageBytes);
  *reinterpret_cast<unsigned short*>(sH + off) = static_cast<unsigned short>(pack_f16x2_sat(v, 0.f) & 0xFFFFu);
}
// element `idx` (of dv row-varying inputs) with value v, under the layer-0 split scheme; the parts of the split
// operand start at multiples of dvp = round_up(dv, 8) so that 8 consecutive inputs are one 16-byte chunk
__device__ __forceinline__ void a0_put(uint8_t* sH, int row, int idx, int dvp, int split, float v) {
  if (split == 4) { a0_store_f16(sH, row, idx, v); return; }
  const float hi = bf16_round(v);
  a0_store(sH, row, idx, hi);
  if (split >= 2) a0_store(sH, row, dvp + idx, v - hi);
  if (split >= 3) a0_store(sH, row, 2 * dvp + idx, hi);
}
// eight consecutive inputs idx0 .. idx0+7 (idx0 % 8 == 0): one 16-byte swizzled store per split part
__device__ __forceinline__ void a0_put8(uint8_t* sH, int row, int idx0, int dvp, int split, const float* v) {
  uint8_t* rowp0 = sH + (row >> 3) * 1024 + (row & 7) * 128;
  if (split == 4) {
    st_shared_v4(rowp0 + (idx0 >> 6) * kStageBytes + ((((idx0 & 63) >> 3) ^ (row & 7)) << 4),
                 pack_f16x2_sat(v[0], v[1]), pack_f16x2_sat(v[2], v[3]), pack_f16x2_sat(v[4], v[5]),
                 pack_f16x2_sat(v[6], v[7]));
    return;
  }
  float hi[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) hi[e] = bf16_round(v[e]);
  const uint32_t h0 = pack_bf16x2(hi[0], hi[1]), h1 = pack_bf16x2(hi[2], hi[3]), h2 = pack_bf16x2(hi[4], hi[5]),
                 h3 = pack_bf16x2(hi[6], hi[7]);
  uint8_t* rowp = sH + (row >> 3) * 1024 + (row & 7) * 128;
  auto chunk_ptr = [&](int k) { return rowp + (k >> 6) * kStageBytes + ((((k & 63) >> 3) ^ (row & 7)) << 4); };
  st_shared_v4(chunk_ptr(idx0), h0, h1, h2, h3);
  if (split >= 2)
    st_shared_v4(chunk_ptr(dvp + idx0), pack_bf16x2(v[0] - hi[0], v[1] - hi[1]), pack_bf16x2(v[2] - hi[2], v[3] - hi[3]),
                 pack_bf16x2(v[4] - hi[4], v[5] - hi[5]), pack_bf16x2(v[6] - hi[6], v[7] - hi[7]));
  if (split >= 3) st_shared_v4(chunk_ptr(2 * dvp + idx0), h0, h1, h2, h3);
}

// Timeline hook (debug): each instrumented thread of CTA 0 owns a quarter of the buffer and appends
// (clock64 << 16 | code) with plain stores — no atomics, so the probe costs a few cycles, not an L2 round trip.
struct TlRole {
  unsigned long long* p;
  unsigned int n, cap;
  bool minimal;   // DMIP_DBG bit 64: record only the pass boundaries (a probe costs ~90 cycles: clock64 is slow)
};
__device__ __forceinline__ TlRole tl_role(const TcParams& P, int dbg, int role, bool on) {
  TlRole r;
  r.p = nullptr;
  r.n = 0;
  r.cap = 0;
  r.minimal = (dbg & 64) != 0;
  if (P.tl != nullptr && blockIdx.x == 0 && on) {
    const int seg = P.tl_cap / 4;
    r.p = P.tl + static_cast<size_t>(role) * seg;
    r.cap = static_cast<unsigned int>(seg - 1);
  }
  return r;
}
__device__ __forceinline__ void tl_mark_impl(TlRole& r, uint32_t code) {
  if (r.p != nullptr && r.n < r.cap && (!r.minimal || code == 0xD00u || (code & 0xF00u) == 0x100u || code == 0xE00u)) {
    r.p[1 + r.n] = (static_cast<unsigned long long>(clock64()) << 16) | code;
    ++r.n;
  }
}
__device__ __forceinline__ void tl_finish_impl(const TlRole& r) {
  if (r.p != nullptr) r.p[0] = r.n;
}
#ifdef DMIP_DEBUG
#define tl_mark(r, code) tl_mark_impl(r, code)
#define tl_finish(r) tl_finish_impl(r)
#define job_mark(r, code) ((void)0)
#elif defined(DMIP_JOBMARKS)
// production code path + four probes per accumulator job (~90 cycles each): -DDMIP_JOBMARKS timing builds
#define tl_mark(r, code) ((void)0)
#define tl_finish(r) tl_finish_impl(r)
#define job_mark(r, code) tl_mark_impl(r, code)
#else
#define tl_mark(r, code) ((void)0)
#define tl_finish(r) ((void)0)
#define job_mark(r, code) ((void)0)
#endif

// ------------------------------------------------------------------------------------------------ the kernel
// NP = 8-column pieces of the fp32 state per particle (xdim <= 8 NP); a row thread keeps ceil(NP / 4) of them.
// VAR = sampler variant (DMIP_CDE also serves the forward mode): decides which per-thread state exists at all.
// L0TMEM = the layer-0 operand is one f16 part in tensor memory (TcNetDev::l0_tmem, the same for every net of the launch);
// otherwise it is built in shared memory.  A compile-time choice, so that each instantiation carries only one builder.
template <int NP, int VAR, bool L0TMEM>
__global__ void __launch_bounds__(kThreads, 1) k_tc_mlp(const __grid_constant__ TcParams P) {
  constexpr int kOwn = (NP + 3) / 4;
  constexpr bool cdiffe = (VAR == DMIP_CDIFFE);
  constexpr bool dps = (VAR == DMIP_DPS);
  extern __shared__ __align__(1024) uint8_t smem[];   // no static shared memory in this kernel: the window base
  if ((smem_u32(smem) & 1023u) != 0u) __trap();       // itself is the swizzle-atom (1024 B) aligned address
  uint8_t* sH = smem + kOffH;
  uint8_t* sB = smem + kOffB;
  float* sB0 = reinterpret_cast<float*>(smem + kOffB0);
  float* sB3 = reinterpret_cast<float*>(smem + kOffB3);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(smem + kOffTmem);
  Bars B;
  B.full = bars;
  B.empty = bars + kNumPairs;
  B.acc_full = bars + 2 * kNumPairs;
  B.acc_empty = B.acc_full + 2;
  B.out_full = B.acc_empty + 2;
  B.out_empty = B.out_full + 1;
  B.sh_free = B.out_empty + 1;
  B.hready = B.sh_free + 1;
  B.a0_ready = B.hready + 4;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // warp-uniform for the compiler
  const int lane = threadIdx.x & 31;

  // ---- one-time setup
  if (warp == kProducerWarp && lane == 0) {
    for (int i = 0; i < kNumPairs; ++i) {
      mbar_init(&B.full[i], 1);
      mbar_init(&B.empty[i], static_cast<uint32_t>(kCluster));   // one tcgen05.commit per CTA of the cluster
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&B.acc_full[i], 1);
      mbar_init(&B.acc_empty[i], kNumRowWarps);
    }
    mbar_init(B.out_full, 1);
    mbar_init(B.out_empty, kNumRowWarps);
    mbar_init(B.sh_free, 1);
    for (int i = 0; i < 4; ++i) mbar_init(&B.hready[i], kNumRowWarps);
    mbar_init(B.a0_ready, kNumRowWarps);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc<kTmemCols>(tmem_holder);
  // zero the activation region once: layer-0 K padding must be finite (it meets zero weights)
  for (int i = threadIdx.x; i < kHBytes / 16; i += kThreads) reinterpret_cast<uint4*>(sH)[i] = make_uint4(0, 0, 0, 0);
  for (int i = threadIdx.x; i < 128; i += kThreads) {
    if (dps) sB3[i] = i < 16 ? P.net[i >> 3].b3[i & 7] : 0.f;
    else sB3[i] = P.net[0].b3[i];   // zero-padded to 128 floats in the packed image
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_holder, 0);   // warp-uniform for the compiler

  // Cluster: the C CTAs of a cluster walk the same stage sequence in lock-step; each loads 1/C of every weight
  // stage and multicasts it to all of them, so L2 serves each line once per cluster instead of once per SM.
  constexpr int C = kCluster;
#ifdef DMIP_DEBUG
  // masked with a value read from shared memory so that ptxas cannot re-materialise it from the constant bank
  const int dbg = P.dbg & static_cast<int>(*reinterpret_cast<volatile uint32_t*>(tmem_holder) == 0xFFFFFFFFu ? 0u : 0xFFFFFFFFu);
#else
  // The DMIP_DBG ablation bits and the timeline exist only in -DDMIP_DEBUG builds: a run-time flag costs a constant-bank
  // re-load (~40 cycles) at every use inside the issue loops.  -DDMIP_EXP=<bits> bakes the same bits in at compile time
  // (timing experiments on otherwise unchanged production code): 1 no weight copies, 2 no MMA issue, 8 no epilogue
  // math, 16 no state pre-update.
#ifndef DMIP_EXP
#define DMIP_EXP 0
#endif
  constexpr int dbg = DMIP_EXP;
#endif
  const int n_tiles = keep(static_cast<int>(P.n_tiles));   // < 2^31 tiles (checked on the host)
  const uint32_t crank = C > 1 ? cluster_ctarank() : 0u;
  const uint16_t cmask = static_cast<uint16_t>((1u << C) - 1u);
  if (C > 1) cluster_sync_all();   // every CTA's mbarriers are initialised before any remote arrive / multicast
  const int tile_first = static_cast<int>(blockIdx.x / C) * C;
  const int tile_stride = keep(static_cast<int>(gridDim.x));

  const int n_pass = keep(P.n_nets);
  const int S = keep(P.S);
  const int n_steps = keep((P.mode == kModeSampler) ? S * (1 + P.n_corr) : 1);   // sub-steps: predictor + correctors
  constexpr int n_ring = kNumPairs;

  if (warp >= kNumRowWarps) {
    reg_dealloc<kRegsSmall>();
    if (warp == kProducerWarp) {
      // ============================================================= producer (whole warp, one elected lane issues)
      int s = 0;
      uint32_t ph = 0;
      TlRole tl = tl_role(P, dbg, 0, lane == 0);
      constexpr uint32_t part = kPairBytes / C;
      for (int tb = tile_first; tb < n_tiles; tb += tile_stride) {
        for (int step = 0; step < n_steps; ++step) {
          for (int p = 0; p < n_pass; ++p) {
            const uint8_t* src = keep(P.net[p].stages);
            const int npairs = keep(P.net[p].n_stages >> 1);   // 4 kb0 + 72 blocks: always even
            for (int pr = 0; pr < npairs; ++pr) {
              mbar_wait(&B.empty[s], ph ^ 1u, 0x100 + s);   // pair s released by the MMA warps of ALL cluster CTAs
              tl_mark(tl, 0x600u | (pr & 0xFF));
              const uint8_t* g = src + static_cast<size_t>(pr) * kPairBytes;
              if (elect_one()) {
                if (dbg & 1) {
                  mbar_arrive(&B.full[s]);
                } else {
                  mbar_arrive_expect_tx(&B.full[s], kPairBytes);
                  if (C == 1)
                    bulk_g2s(sB + s * kPairBytes, g, kPairBytes, &B.full[s]);
                  else
                    bulk_g2s_multicast(sB + s * kPairBytes + crank * part, g + crank * part, part, &B.full[s], cmask);
                }
              }
              __syncwarp();
              if (++s == n_ring) { s = 0; ph ^= 1u; }
            }
          }
        }
      }
      tl_finish(tl);
    } else if (warp == kMmaWarp) {
      // ============================================================= MMA issuer (whole warp, one elected lane issues)
      // The tensor core queues only about one instruction ahead of the issuing thread, so every cycle this loop spends
      // between two MMAs beyond ~1 MMA duration is a cycle the tensor pipe idles: the loop is kept to the bare
      // sequence  wait(pair) / 8 x (descriptor add, UTCHMMA) / commit  with all addressing as immediates.
      int s = 0;             // ring pair being consumed
      uint32_t ph = 0;
      uint32_t job = 0;
      uint32_t hr_par = 0;   // bit c = parity of hready[c]
      uint32_t a0_par = 0;
      uint32_t ch0 = 0, ch1 = 0, n_out = 0;          // hidden uses of accumulator buffer 0/1; output jobs so far
      uint32_t lastkind = 0;                         // 2 bits per buffer: 0 never used, 1 hidden job, 2 output job
      uint32_t blk = 0;                              // 16 KB weight blocks consumed by layer 0 of this pass
      TlRole tl = tl_role(P, dbg, 1, lane == 0);
      const uint32_t a_base = (smem_u32(sH) & 0x3FFFFu) >> 4;    // descriptor address fields (16-byte units)
      const uint32_t b_base = (smem_u32(sB) & 0x3FFFFu) >> 4;
      const uint64_t desc_hi = umma_smem_desc_sw128(0) & 0xFFFFFFFF00000000ull;   // everything but the address field
      constexpr uint32_t kBlk16 = kStageBytes >> 4, kPair16 = kPairBytes >> 4;

      // wait until the accumulator buffer's previous user has drained it, then book this use
      auto acquire_acc = [&](int buf, bool is_out, int jl) {
        const uint32_t lk = (lastkind >> (2 * buf)) & 3u;
        tl_mark(tl, 0xB00u | jl);
        if (lk == 1u) mbar_wait(&B.acc_empty[buf], ((buf ? ch1 : ch0) - 1u) & 1u, 0x300 + buf);
        else if (lk == 2u) mbar_wait(B.out_empty, (n_out - 1u) & 1u, 0x310 + buf);   // = the latest output job
        tl_mark(tl, 0x100u | jl);
        job_mark(tl, 0x100u | jl);
        if (is_out) ++n_out; else { if (buf) ++ch1; else ++ch0; }
        lastkind = (lastkind & ~(3u << (2 * buf))) | ((is_out ? 2u : 1u) << (2 * buf));
      };

      for (int tb = tile_first; tb < n_tiles; tb += tile_stride) {
        for (int step = 0; step < n_steps; ++step) {
          for (int p = 0; p < n_pass; ++p) {
            const int net_kb0 = keep(P.net[p].kb0), net_ksteps0 = keep(P.net[p].ksteps0);
            const uint32_t idesc_out = umma_idesc_bf16(128, static_cast<uint32_t>(keep(P.net[p].outpad)));
            constexpr uint32_t idesc_hid = umma_idesc_bf16(128, 128);
            const uint32_t idesc_l0 = keep(P.net[p].l0_f16) ? umma_idesc_f16(128, 128) : idesc_hid;
            tl_mark(tl, 0xD00u);
            job_mark(tl, 0xD00u);
            mbar_wait(B.a0_ready, a0_par, 0x200);
            tl_mark(tl, 0xE00u);
            a0_par ^= 1u;
            int jl = 0;
            // ---- layer 0: A0 (shared memory) x W0 chunks; K = 16 ksteps0 is arbitrary, blocks may straddle ring pairs
            blk = 0;
#pragma unroll 1
            for (int c = 0; c < 4; ++c, ++job, ++jl) {
              const int buf = job & 1;
              acquire_acc(buf, false, jl);
              const uint32_t d_tmem = tmem_base + kTmemAcc + buf * 128;
#pragma unroll 1
              for (int kb = 0; kb < net_kb0; ++kb, ++blk) {
                const uint32_t half = blk & 1u;   // which 16 KB slot of the pair
                if (half == 0u) mbar_wait(&B.full[s], ph, 0x500 + s);
                tc_fence_after();
                const int nk = (kb == net_kb0 - 1) ? (net_ksteps0 - 4 * (net_kb0 - 1)) : 4;
                const uint32_t b_lo = b_base + s * kPair16 + half * kBlk16;
                const uint32_t a_lo = a_base + kb * kBlk16;
                if (elect_one()) {
                  if (!(dbg & 2)) {
                    if (L0TMEM) {
                      const uint32_t a_tm = tmem_base + kTmemL0 + kb * 32;
#pragma unroll
                      for (int kk = 0; kk < 4; ++kk)
                        if (kk < nk) umma_ts(d_tmem, a_tm + kk * 8, desc_hi | (b_lo + kk * 2), idesc_l0, (kb | kk) != 0 ? 1u : 0u);
                    } else {
#pragma unroll
                      for (int kk = 0; kk < 4; ++kk)
                        if (kk < nk)
                          umma_ss(d_tmem, desc_hi | (a_lo + kk * 2), desc_hi | (b_lo + kk * 2), idesc_l0, (kb | kk) != 0 ? 1u : 0u);
                    }
                  }
                  if (half == 1u) tc_commit_multicast(&B.empty[s], cmask);
                  if (kb == net_kb0 - 1) tc_commit(&B.acc_full[buf]);
                }
                __syncwarp();
                if (half == 1u) { if (++s == n_ring) { s = 0; ph ^= 1u; } }
              }
              tl_mark(tl, 0x200u | jl);
              job_mark(tl, 0x200u | jl);
            }
            // ---- layers 1..3: K = 512 = 4 ring pairs per chunk, pair-aligned (layer 0 consumed 4 kb0 blocks)
#pragma unroll 1
            for (int l = 1; l < 4; ++l) {
              const int n_chunks = (l == 3) ? 1 : 4;
#ifndef DMIP_H_F16
              const uint32_t idesc = (l == 3) ? idesc_out : idesc_hid;
#else
              const uint32_t idesc = ((l == 3) ? idesc_out : idesc_hid) & ~((7u << 7) | (7u << 10));   // H_l, W_l: f16 (format 0)
#endif
#pragma unroll 1
              for (int c = 0; c < n_chunks; ++c, ++job, ++jl) {
                const int buf = job & 1;
                acquire_acc(buf, l == 3, jl);
                const uint32_t d_tmem = tmem_base + kTmemAcc + buf * 128;
#pragma unroll 1
                for (int pr = 0; pr < 4; ++pr) {
                  if (c == 0) {   // K-blocks 2 pr, 2 pr + 1 of this layer's A operand come from chunk pr of the previous epilogue
                    mbar_wait(&B.hready[pr], (hr_par >> pr) & 1u, 0x400 + pr);
                    hr_par ^= 1u << pr;
                  }
                  mbar_wait(&B.full[s], ph, 0x500 + s);
                  tc_fence_after();
                  const uint32_t b_lo = b_base + s * kPair16;
                  if (elect_one()) {
                    if (!(dbg & 2)) {
                      if (l == 2 && !(kL2TailTmem && pr == 3)) {   // A = H2 in shared memory
                        const uint32_t a_lo = a_base + pr * kPair16;
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                          umma_ss(d_tmem, desc_hi | (a_lo + (j >> 2) * kBlk16 + (j & 3) * 2),
                                  desc_hi | (b_lo + (j >> 2) * kBlk16 + (j & 3) * 2), idesc, (pr | j) != 0 ? 1u : 0u);
                      } else {               // A = H1 / H3 (and the last quarter of H2) in tensor memory
                        const uint32_t a_tm = tmem_base + kTmemH + pr * 64;
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                          umma_ts(d_tmem, a_tm + j * 8, desc_hi | (b_lo + (j >> 2) * kBlk16 + (j & 3) * 2), idesc,
                                  (pr | j) != 0 ? 1u : 0u);
                      }
                    }
                    tc_commit_multicast(&B.empty[s], cmask);
                    if (pr == 3) {
                      if (l == 3) tc_commit(B.out_full);
                      else tc_commit(&B.acc_full[buf]);
                      if (l == 2 && c == 3) tc_commit(B.sh_free);
                    }
                  }
                  __syncwarp();
                  if (++s == n_ring) { s = 0; ph ^= 1u; }
                }
                tl_mark(tl, 0x200u | jl);
                job_mark(tl, 0x200u | jl);
              }
            }
          }
        }
      }
      tl_finish(tl);
    }
  } else {
    // =============================================================== row warps (512 threads, 4 per particle row)
    reg_alloc<kRegsRow>();
    const int quarter = warp & 3;  // warp % 4: the TMEM lane quarter this warp may access
    const int cgp = warp >> 2;     // column group: 32 of a chunk's 128 columns; a quarter of the state pieces
    const int row = quarter * 32 + lane;
    const int et = threadIdx.x;    // 0..511: owner of hidden unit `et` of the effective layer-0 bias
    const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    if (L0TMEM && cgp == 0) {
      // K padding of the tensor-memory layer-0 operand must be finite from the first step on (it meets zero weights)
      const uint32_t z[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int c0 = 0; c0 < 64; c0 += 16) tmem_st16(lane_taddr + kTmemL0 + c0, z);
      tc_wait_st();
    }
    asm volatile("bar.sync 2, 512;" ::: "memory");   // row warps only: zeros before any operand piece is written
    TlRole tl = tl_role(P, dbg, warp == 0 ? 2 : 3, lane == 0 && (warp == 0 || warp == 12));
    uint32_t job = 0;     // global job counter (13 per pass; accumulator buffer = job & 1)
    uint32_t npass = 0;   // running pass counter: layer-0 bias buffer, parity of the once-per-pass barriers
    uint32_t cf0 = 0, cf1 = 0;   // hidden chunks seen in accumulator buffer 0 / 1
    const SdeSched sch = {P.sde_kind, S, P.n_corr, P.T, P.bmin, P.bmax, P.snr, P.delta, P.sqrt_delta};
    const TcNetDev& net_last = P.net[n_pass - 1];
    const int dvp = (net_last.dv + 7) & ~7;
    const int split = P.net[0].l0_f16 ? 4 : P.net[0].split;   // 4: one f16 part (a0_put / a0_put8)
    constexpr bool l0_tmem = L0TMEM;
    const bool sampler = (P.mode == kModeSampler);
    const int xdim = P.xdim;
    // state pieces (8 columns) of this row owned by this thread: [piece_lo, piece_lo + n_own)
    const int np = sampler ? (xdim + 7) >> 3 : 0;
    const int pbase = np >> 2, prem = np & 3;
    const int n_own = pbase + (cgp < prem ? 1 : 0);
    const int piece_lo = cgp * pbase + (cgp < prem ? cgp : prem);
    float xs[kOwn * 8];   // fp32 SDE state
    float yt[cdiffe ? 8 : 1];   // CDiffE: re-diffused observation columns 4 cgp .. +3 and 4 (cgp + 4) .. +3 of the next step
    float myU[2], myWt[2];      // [1] is used by DPS only
#pragma unroll
    for (int j = 0; j < kOwn * 8; ++j) xs[j] = 0.f;
#pragma unroll
    for (int j = 0; j < (cdiffe ? 8 : 1); ++j) yt[j] = 0.f;
    myU[0] = myU[1] = myWt[0] = myWt[1] = 0.f;

    for (int tb = tile_first; tb < n_tiles; tb += tile_stride) {
      // a cluster whose last round has fewer tiles than CTAs still runs every CTA (lock-step), on masked rows
      const bool tile_ok = tb + static_cast<int>(crank) < n_tiles;
      const int tile = tile_ok ? tb + static_cast<int>(crank) : n_tiles - 1;
      const int obs = static_cast<int>(tile / P.tiles_per_obs);
      const long long prow = static_cast<long long>(tile % P.tiles_per_obs) * kTileM + row;
      const bool valid = tile_ok && prow < P.n_per_obs;
      const long long grow = static_cast<long long>(obs) * P.n_per_obs + prow;
      const unsigned long long gidx = P.gidx_base + static_cast<unsigned long long>(grow);

      // y_t = alpha(tau) y + std(tau) eta   (sdes.py:37-49 via models/diffusion.py:172): quads cgp and cgp + 4
      auto diffuse_y = [&](int stp) {
        if (!cdiffe) return;
        float g2u, alpha, var;
        sde_terms<true>(sch, sde_substep_tau(sch, stp), g2u, alpha, var);
        const float sd = sqrtf(var);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int q = cgp + 4 * h;
          if (q * 4 < P.ydim) {
            float z[4] = {0.f, 0.f, 0.f, 0.f};
            if (P.rng_mode == DMIP_RNG_PHILOX) philox_normal4(gidx, pin_here(static_cast<uint32_t>(stp)), kStreamObs, q, P.seed, z);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int jj = q * 4 + e;
              float v = 0.f;
              if (valid && jj < P.ydim) {
                const float eta = P.rng_mode == DMIP_RNG_PHILOX
                                      ? z[e]
                                      : P.ynoise[(static_cast<long long>(stp) * (static_cast<long long>(P.n_obs) * P.n_per_obs) + grow) * P.ydim + jj];
                v = fmaf(sd, eta, alpha * P.y[obs * P.ydim + jj]);
              }
              yt[cdiffe ? h * 4 + e : 0] = v;
            }
          }
        }
      };
      auto put_yt = [&]() {
        if (!cdiffe) return;
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int jj = (cgp + 4 * h) * 4 + e;
            if (jj < P.ydim) a0_put(sH, row, xdim + jj, dvp, split, yt[cdiffe ? h * 4 + e : 0]);
          }
      };
      // layer-0 operand columns of this thread's state pieces
      auto put_x = [&]() {
#pragma unroll
        for (int i = 0; i < kOwn; ++i) {
          if (i < n_own) {
            const int pc = piece_lo + i;
            if (l0_tmem) {   // one f16 part in tensor memory: 8 elements = 4 columns of this row's lane
              const float* v = &xs[i * 8];
              tmem_st4(lane_taddr + kTmemL0 + static_cast<uint32_t>(pc * 4), pack_f16x2_sat(v[0], v[1]),
                       pack_f16x2_sat(v[2], v[3]), pack_f16x2_sat(v[4], v[5]), pack_f16x2_sat(v[6], v[7]));
            } else if (cdiffe) {   // the columns right after x hold y_t: touch only the x elements
#pragma unroll
              for (int e = 0; e < 8; ++e)
                if (pc * 8 + e < xdim) a0_put(sH, row, pc * 8 + e, dvp, split, xs[i * 8 + e]);
            } else {
              a0_put8(sH, row, pc * 8, dvp, split, &xs[i * 8]);
            }
          }
        }
      };

      // operand written: make it visible to the tensor core (shared-memory operand: async-proxy fence; tensor-memory
      // operand: the stores have landed) and tell the issuer
      auto publish_a0 = [&]() {
        if (l0_tmem) {
          tc_wait_st();
          tc_fence_before();
        } else {
          fence_proxy_async_smem();
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(B.a0_ready);
      };

      // ---- tile init
      if (sampler) {
        // per-observation parts of the effective layer-0 bias of hidden unit `et`
        for (int p = 0; p < n_pass; ++p) {
          const TcNetDev& net = P.net[p];
          float u = net.b0[et];
          const float* wr = net.w0c + static_cast<size_t>(et) * net.n_const;
          for (int j = 0; j + 1 < net.n_const; ++j) u = fmaf(wr[j], P.y[obs * P.ydim + j], u);
          const float wt = wr[net.n_const - 1];
          if (p == 0) { myU[0] = u; myWt[0] = wt; } else if (dps) { myU[1] = u; myWt[1] = wt; }
          if (p == 0) sB0[et] = fmaf(sde_substep_tau(sch, 0), wt, u);   // the previous tile's last pass has drained it
        }
#pragma unroll
        for (int i = 0; i < kOwn; ++i) {
          if (i < n_own) {
            const int pc = piece_lo + i;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              float z4[4] = {0.f, 0.f, 0.f, 0.f};
              if (P.rng_mode == DMIP_RNG_PHILOX) philox_normal4(gidx, kPhiloxStepInit, kStreamState, pc * 2 + h, P.seed, z4);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int j = pc * 8 + h * 4 + e;
                float v = 0.f;
                if (valid && j < xdim) {
                  const float zz = P.rng_mode == DMIP_RNG_PHILOX ? z4[e] : P.x0[grow * xdim + j];
                  v = zz * P.std + P.mean;   // models/diffusion.py:32-33
                }
                xs[i * 8 + h * 4 + e] = v;
              }
            }
          }
        }
        put_x();
        if (cdiffe) {
          diffuse_y(0);
          put_yt();
        }
      } else {
        const TcNetDev& net = P.net[0];
        sB0[et] = net.b0[et];
        if (valid) {
          for (int k = cgp; k < net.dv; k += 4) {
            float v;
            if (k < P.fx_dim) v = P.fx[grow * P.fx_dim + k];
            else if (k < P.fx_dim + P.fcond_dim) v = P.fcond[grow * P.fcond_dim + (k - P.fx_dim)];
            else v = P.ft[grow];
            a0_put(sH, row, k, dvp, split, v);
          }
        }
      }
      publish_a0();
      tl_mark(tl, 0x500u);

      for (int step = 0; step < n_steps; ++step) {
        const SdeCoef co = sde_coef<true>(sch, step, dps);   // x <- x (1 + kx) + ke eps + ca net   at time co.tau
        const float tau = co.tau;
        const bool last_step = (step == n_steps - 1);
        float stash[dps ? 8 : 1];   // DPS: prior-net output of this step
#pragma unroll
        for (int e = 0; e < (dps ? 8 : 1); ++e) stash[e] = 0.f;

        for (int p = 0; p < n_pass; ++p, ++npass) {
          const TcNetDev& net = P.net[p];
          const bool last_pass = (p == n_pass - 1);
          const bool fuse_draw = sampler && last_pass && !(dbg & 16) && P.rng_mode == DMIP_RNG_PHILOX;
          float zdraw[4] = {0.f, 0.f, 0.f, 0.f}, zdraw4[4] = {0.f, 0.f, 0.f, 0.f};   // noise of the piece updated after chunk c
          // ---- layers 0..2
          int jl = 0;
#pragma unroll 1
          for (int l = 0; l < 3; ++l) {
            const float* bias = (l == 0) ? sB0 : (l == 1 ? net.b1 : net.b2);
#pragma unroll 1
            for (int c = 0; c < 4; ++c, ++job, ++jl) {
              const int buf = job & 1;
              job_mark(tl, 0x600u | jl);
              mbar_wait(&B.acc_full[buf], (buf ? cf1 : cf0) & 1u, 0x800 + buf);
              if (buf) ++cf1; else ++cf0;
              tc_fence_after();
              tl_mark(tl, 0x300u | jl);
              job_mark(tl, 0x300u | jl);
              const uint32_t acc_col = kTmemAcc + buf * 128;
              if (dbg & 8) {   // debug: no epilogue work at all, only the handshakes
                tc_fence_before();
                __syncwarp();
                if (lane == 0) { mbar_arrive(&B.acc_empty[buf]); mbar_arrive(&B.hready[c]); }
              } else if (l == 0)
                epi_hidden<true, true>(lane_taddr, acc_col, cgp, row, c, lane, bias, sH, &B.acc_empty[buf], &B.hready[c]);
              else {
                // State piece i is drawn and pre-updated at chunk (l, c) = (1 + i/2, 2 (i%2)): never in two consecutive
                // chunks and never in a layer's last chunk, whose epilogue the next layer's MMAs are waiting for.
                const int ip = (l - 1) * 2 + (c >> 1);
                const bool draw_here = fuse_draw && (c & 1) == 0 && ip < kOwn;
                const int pc = piece_lo + ip;
                // the Philox / Box-Muller draw rides inside the epilogue's instruction stream
                auto draw = [&]() {
                  const uint32_t here = pin_here(static_cast<uint32_t>(step));
                  philox_normal4(gidx, here, kStreamState, pc * 2, P.seed, zdraw);
                  philox_normal4(gidx, here, kStreamState, pc * 2 + 1, P.seed, zdraw4);
                };
                if (l == 1 && !(kL2TailTmem && c == 3)) {
                  if (draw_here)
                    epi_hidden<false, false>(lane_taddr, acc_col, cgp, row, c, lane, bias, sH, &B.acc_empty[buf], &B.hready[c], draw);
                  else
                    epi_hidden<false, false>(lane_taddr, acc_col, cgp, row, c, lane, bias, sH, &B.acc_empty[buf], &B.hready[c]);
                } else {
                  if (draw_here)
                    epi_hidden<false, true>(lane_taddr, acc_col, cgp, row, c, lane, bias, sH, &B.acc_empty[buf], &B.hready[c], draw);
                  else
                    epi_hidden<false, true>(lane_taddr, acc_col, cgp, row, c, lane, bias, sH, &B.acc_empty[buf], &B.hready[c]);
                }
              }
              tl_mark(tl, 0x400u | jl);
              job_mark(tl, 0x400u | jl);
              if (sampler && last_pass && !(dbg & 16)) {
                if (l >= 1 && (c & 1) == 0) {
                  // ---- in the shadow of the MMA-bound layers, one state piece per accumulator chunk: the part of the
                  // Euler–Maruyama update that does not need the net output,
                  //   x <- x + delta*beta/2*x + sqrt(delta*beta)*eps            (models/diffusion.py:42, sdes.py:77-87)
#pragma unroll
                  for (int i = 0; i < kOwn; ++i) {
                    if (i == (l - 1) * 2 + (c >> 1) && i < n_own) {
                      const int pc = piece_lo + i;
                      // the output layer's bias joins here too (x += ca * b3), off the step boundary's critical path
                      const float ca = co.ca;
                      const float* b3s = sB3 + (dps ? 8 : pc * 8);   // DPS: one piece, the likelihood net's bias
                      const float4 q0 = *reinterpret_cast<const float4*>(b3s);
                      const float4 q1 = *reinterpret_cast<const float4*>(b3s + 4);
                      const float b3v[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
                      // The draw itself was made inside this chunk's epilogue (fuse_draw); pin_here ties it to that
                      // point of the schedule: the generator only depends on (particle, step, piece), and the compiler
                      // otherwise hoists ALL of a step's draws to the top of the step — 7800 cycles in front of the
                      // layer-0 epilogue instead of in the MMAs' shadow.
                      float za[4], zb[4];
#pragma unroll
                      for (int e = 0; e < 4; ++e) { za[e] = zdraw[e]; zb[e] = zdraw4[e]; }
                      float eps[8];
#pragma unroll
                      for (int e = 0; e < 8; ++e) {
                        const int j = pc * 8 + e;
                        eps[e] = 0.f;
                        if (valid && j < xdim)
                          eps[e] = fuse_draw ? (e < 4 ? za[e & 3] : zb[e & 3])
                                             : P.noise[(static_cast<long long>(step) * (static_cast<long long>(P.n_obs) * P.n_per_obs) + grow) * xdim + j];
                      }
                      // x <- fmaf(kx, x, x) + fmaf(ke, eps, ca * b3) on packed pairs, in that operation order
                      const unsigned long long kx2 = f32x2_pack(co.kx, co.kx), ke2 = f32x2_pack(co.ke, co.ke),
                                               ca2 = f32x2_pack(ca, ca);
#pragma unroll
                      for (int e = 0; e < 8; e += 2) {
                        const unsigned long long x2 = f32x2_pack(xs[i * 8 + e], xs[i * 8 + e + 1]);
                        const unsigned long long n2 =
                            f32x2_fma(ke2, f32x2_pack(eps[e], eps[e + 1]), f32x2_mul(ca2, f32x2_pack(b3v[e], b3v[e + 1])));
                        f32x2_unpack(f32x2_add(f32x2_fma(kx2, x2, x2), n2), xs[i * 8 + e], xs[i * 8 + e + 1]);
                      }
                    }
                  }
                }
                if (l == 2 && c == 1 && cdiffe && !last_step) diffuse_y(step + 1);
              }
            }
          }
          // ---- layer 2 has consumed the shared-memory operand region: operand columns that do not depend on this
          // pass's output can be written now
          tl_mark(tl, 0x310u);
          mbar_wait(B.sh_free, npass & 1u, 0x600);
          if (sampler) {
            // layer 2 is done, so every row warp has left this pass's layer-0 epilogue: the single bias buffer may take
            // the next pass's effective layer-0 bias  b0 + W0[:,y]·y + tau'·W0[:,t]
            const bool wrap = (p + 1 == n_pass);
            const float tau_n = wrap ? sde_substep_tau(sch, step + 1) : tau;
            const float u = (wrap || !dps) ? myU[0] : myU[1];
            const float wt = (wrap || !dps) ? myWt[0] : myWt[1];
            sB0[et] = fmaf(tau_n, wt, u);
          }
          if (sampler) {
            if (!last_pass && !l0_tmem) {
              put_x();   // DPS: same x for the likelihood net (H2 overwrote the operand)
              publish_a0();
            } else if (cdiffe && !last_step) {
              put_yt();
            }
          }
          // ---- output layer
          tl_mark(tl, 0x320u);
          mbar_wait(B.out_full, npass & 1u, 0x700);
          tc_fence_after();
          tl_mark(tl, 0x300u | 12);
          job_mark(tl, 0x300u | 12);
          const uint32_t acc_col = kTmemAcc + (job & 1u) * 128;
          ++job;
          if (!sampler) {
            const float* b3 = net.b3;   // zero-padded to 128 floats in the packed image
            for (int pc = cgp; pc * 8 < P.out_dim; pc += 4) {
              uint32_t v[8];
              tmem_ld8(lane_taddr + acc_col + pc * 8, v);
              tc_wait_ld();
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int j = pc * 8 + e;
                if (valid && j < P.out_dim) P.out[grow * P.out_dim + j] = __uint_as_float(v[e]) + b3[j];
              }
            }
          } else if (!last_pass) {
            if (n_own > 0) {   // DPS prior pass: xdim <= 8, the single piece belongs to column group 0
              uint32_t v[8];
              tmem_ld8(lane_taddr + acc_col, v);
              tc_wait_ld();
#pragma unroll
              for (int e = 0; e < 8; ++e) stash[dps ? e : 0] = __uint_as_float(v[e]) + sB3[e];
            }
            if (l0_tmem) {   // the prior pass's output layer has read all of H3: its last columns take x again
              put_x();
              publish_a0();
            }
          } else {
            // CDE/CDiffE: mu = sqrt(beta) a + beta x / 2 (sdes.py:77-79, Q3);
            // DPS: a = sqrt(beta) (prior + lik) (nets.py:155-157)  =>  mu = beta (prior + lik) + beta x / 2.
            // The bias b3 is already in x (pre-update).  No masks: padded columns meet zero weights and zero noise and
            // stay zero; rows past the end of the tile integrate a harmless deterministic path and are never written.
            const unsigned long long ca2 = f32x2_pack(co.ca, co.ca);
            uint32_t v[kOwn][8];
#pragma unroll
            for (int i = 0; i < kOwn; ++i)
              if (i < n_own) tmem_ld8(lane_taddr + acc_col + (piece_lo + i) * 8, v[i]);
            tc_wait_ld();
#pragma unroll
            for (int i = 0; i < kOwn; ++i) {
              if (i < n_own) {
#pragma unroll
                for (int e = 0; e < 8; e += 2) {   // x <- fmaf(ca, a, x) on packed pairs
                  unsigned long long a2 = f32x2_pack(__uint_as_float(v[i][e]), __uint_as_float(v[i][e + 1]));
                  if (dps) a2 = f32x2_add(a2, f32x2_pack(stash[dps ? e : 0], stash[dps ? e + 1 : 0]));
                  f32x2_unpack(f32x2_fma(ca2, a2, f32x2_pack(xs[i * 8 + e], xs[i * 8 + e + 1])), xs[i * 8 + e],
                               xs[i * 8 + e + 1]);
                }
              }
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(B.out_empty);
          tl_mark(tl, 0x400u | 12);
          job_mark(tl, 0x400u | 12);
          if (sampler && last_pass) {
            if (last_step) {
              if (valid) {
#pragma unroll
                for (int i = 0; i < kOwn; ++i)
                  if (i < n_own) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                      const int j = (piece_lo + i) * 8 + e;
                      if (j < xdim) P.out[grow * xdim + j] = xs[i * 8 + e];
                    }
                  }
              }
            } else {
              put_x();   // next step's layer-0 operand
              publish_a0();
              tl_mark(tl, 0x500u);
              job_mark(tl, 0x500u);
            }
          }
        }  // pass
      }    // step
    }      // tile
    tl_finish(tl);
  }

  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (C > 1) cluster_sync_all();   // no CTA leaves while a peer may still signal its barriers
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc<kTmemCols>(tmem_base);
  }
}

int fill_net(const DmipMlp* net, const void* packed, int n_varying, int out_rows, int split, TcNetDev* o) {
  TcNetGeom g;
  int rc = tc_net_geom(net, n_varying, out_rows, split, &g);
  if (rc) return rc;
  const uint8_t* base = static_cast<const uint8_t*>(packed);
  const float* tail = reinterpret_cast<const float*>(base + g.stage_bytes());
  o->stages = base;
  o->b0 = tail;
  o->b1 = tail + 512;
  o->b2 = tail + 1024;
  o->b3 = tail + 1536;
  o->w0c = tail + 1664;
  o->kb0 = g.kb0;
  o->ksteps0 = g.k0pad / 16;
  o->dv = g.n_varying;
  o->split = g.split;
  o->l0_f16 = g.l0_f16;
  o->l0_tmem = 0;
  o->outpad = g.outpad;
  o->n_const = g.n_const;
  o->n_stages = g.n_stages;
  return 0;
}

int g_n_sm = 0;
int g_dbg = 0;
unsigned long long* g_tl = nullptr;
int g_tl_cap = 0;

bool g_dev_ready[64] = {};   // cudaFuncSetAttribute is per device: one process may drive several GPUs

int init_device() {
  int dev = 0;
  DMIP_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !g_dev_ready[dev]) {
    DMIP_CHECK_CUDA(cudaDeviceGetAttribute(&g_n_sm, cudaDevAttrMultiProcessorCount, dev));
#define DMIP_SET_SMEM(NP, VAR, L0TMEM) \
  DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_tc_mlp<NP, VAR, L0TMEM>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes))
    DMIP_SET_SMEM(1, DMIP_CDE, false);
    DMIP_SET_SMEM(1, DMIP_CDE, true);
    DMIP_SET_SMEM(1, DMIP_CDIFFE, false);
    DMIP_SET_SMEM(1, DMIP_DPS, false);
    DMIP_SET_SMEM(1, DMIP_DPS, true);
    DMIP_SET_SMEM(4, DMIP_CDE, false);
    DMIP_SET_SMEM(4, DMIP_CDE, true);
    DMIP_SET_SMEM(4, DMIP_CDIFFE, false);
    DMIP_SET_SMEM(13, DMIP_CDE, false);
    DMIP_SET_SMEM(13, DMIP_CDE, true);
#undef DMIP_SET_SMEM
    if (getenv("DMIP_DBG")) g_dbg = atoi(getenv("DMIP_DBG"));
    if (dev >= 0 && dev < 64) g_dev_ready[dev] = true;
  }
  return DMIP_OK;
}

int launch(TcParams& P, cudaStream_t s) {
  int rc = init_device();
  if (rc) return rc;
  const int n_sm = g_n_sm;
  P.tl = g_tl;
  P.tl_cap = g_tl_cap;
  if (P.n_tiles <= 0) return DMIP_OK;
  DMIP_REQUIRE(P.n_tiles < (1LL << 31), "too many particle tiles in one call (%lld); split the call", P.n_tiles);
  const int C = kCluster;   // a lone tile still launches a pair: the second CTA runs masked rows
  P.cluster = C;
  P.dbg = g_dbg;
  const long long want_clusters = (P.n_tiles + C - 1) / C;
  const long long max_clusters = n_sm / C;   // pairs: all 74 are co-resident (tools/probe/cluster_probe.cu; 4: only 33)
  const long long n_clusters = want_clusters < max_clusters ? want_clusters : max_clusters;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(n_clusters * C));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = static_cast<unsigned>(C);
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const int state_cols = (P.mode == kModeSampler) ? P.xdim : 1;
  const int var = (P.mode == kModeSampler) ? P.variant : DMIP_CDE;
  const bool l0t = P.net[0].l0_tmem != 0;
  for (int p = 1; p < P.n_nets; ++p)
    DMIP_REQUIRE((P.net[p].l0_tmem != 0) == l0t, "all nets of one sampler launch need the same layer-0 operand location");
  if (var == DMIP_DPS) {
    if (l0t) DMIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_tc_mlp<1, DMIP_DPS, true>, P));
    else DMIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_tc_mlp<1, DMIP_DPS, false>, P));
  } else if (var == DMIP_CDIFFE) {   // never l0_tmem: the operand holds y_t next to x
    if (state_cols <= 8) DMIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_tc_mlp<1, DMIP_CDIFFE, false>, P));
    else DMIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_tc_mlp<4, DMIP_CDIFFE, false>, P));
  } else if (l0t) {
    if (state_cols <= 8) DMIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_tc_mlp<1, DMIP_CDE, true>, P));
    else if (state_cols <= 32) DMIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_tc_mlp<4, DMIP_CDE, true>, P));
    else DMIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_tc_mlp<13, DMIP_CDE, true>, P));
  } else {
    if (state_cols <= 8) DMIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_tc_mlp<1, DMIP_CDE, false>, P));
    else if (state_cols <= 32) DMIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_tc_mlp<4, DMIP_CDE, false>, P));
    else DMIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_tc_mlp<13, DMIP_CDE, false>, P));
  }
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return DMIP_OK;
}

}  // namespace

size_t sampler_tc_workspace() {
  return 256;   // the state lives in registers, activations in shared / tensor memory: no device scratch is needed
}

void tcl_debug_set_timeline(unsigned long long* buf, int cap);   // dmip_tcl.cu
void debug_set_timeline(unsigned long long* buf, int cap) {
  g_tl = buf;
  g_tl_cap = cap;
  tcl_debug_set_timeline(buf, cap);
}

int launch_sampler_tc(const DmipSampler* d, cudaStream_t s) {
  TcParams P = {};
  DMIP_REQUIRE(d->xdim <= 104, "tcgen05 sampler keeps the state in registers: xdim <= 104 (got %d); use DMIP_PREC_F32", d->xdim);
  if (d->variant == DMIP_CDIFFE)
    DMIP_REQUIRE(d->xdim <= 32 && d->ydim <= 24, "tcgen05 CDiffE sampler supports xdim <= 32, ydim <= 24 (got %d, %d); "
                 "use DMIP_PREC_F32", d->xdim, d->ydim);
  P.mode = kModeSampler;
  P.variant = d->variant;
  const int dv = d->variant == DMIP_CDIFFE ? d->xdim + d->ydim : d->xdim;
  int rc;
  if (d->variant == DMIP_DPS) {
    P.n_nets = 2;
    DMIP_REQUIRE(d->packed2 != nullptr, "DPS sampler needs packed2 (prior_net image)");
    DMIP_REQUIRE(d->xdim <= 8, "DPS tcgen05 sampler supports xdim <= 8 (got %d)", d->xdim);
    if ((rc = fill_net(&d->net2, d->packed2, d->xdim, d->xdim, d->l0_split, &P.net[0]))) return rc;  // prior (MLP2)
    if ((rc = fill_net(&d->net, d->packed, d->xdim, d->xdim, d->l0_split, &P.net[1]))) return rc;    // likelihood
  } else {
    P.n_nets = 1;
    if ((rc = fill_net(&d->net, d->packed, dv, d->xdim, d->l0_split, &P.net[0]))) return rc;
  }
  // tensor-memory layer-0 operand: one f16 part of <= 128 k, whole 8-element state pieces (CDE / DPS)
  for (int p = 0; p < P.n_nets; ++p)
    P.net[p].l0_tmem = (P.net[p].l0_f16 && d->variant != DMIP_CDIFFE && P.net[p].ksteps0 * 16 <= 128) ? 1 : 0;
  P.xdim = d->xdim;
  P.ydim = d->ydim;
  P.n_obs = d->n_obs;
  P.n_per_obs = d->n_per_obs;
  P.tiles_per_obs = static_cast<int>((d->n_per_obs + kTileM - 1) / kTileM);
  P.n_tiles = static_cast<long long>(P.tiles_per_obs) * d->n_obs;
  P.S = d->num_steps;
  P.T = d->T;
  P.sde_kind = d->sde_kind;
  P.bmin = d->sde_kind == DMIP_SDE_VE ? d->sigma_min : d->beta_min;
  P.bmax = d->sde_kind == DMIP_SDE_VE ? d->sigma_max : d->beta_max;
  P.n_corr = d->n_corrector;
  P.snr = d->snr;
  P.mean = d->mean;
  P.std = d->std;
  const double delta = static_cast<double>(d->T) / d->num_steps;  // models/diffusion.py:31
  P.delta = static_cast<float>(delta);
  P.sqrt_delta = static_cast<float>(sqrt(delta));
  P.y = d->y;
  P.out = d->out;
  P.rng_mode = d->rng_mode;
  P.seed = d->seed;
  P.gidx_base = d->gidx_base;
  P.x0 = d->x0;
  P.noise = d->noise;
  P.ynoise = d->ynoise;
  return launch(P, s);
}

int launch_forward_tc(const DmipForward* d, cudaStream_t s) {
  TcParams P = {};
  P.mode = kModeForward;
  P.variant = DMIP_CDE;
  P.n_nets = 1;
  int rc;
  if ((rc = fill_net(&d->net, d->packed, d->net.in_dim, d->net.out_dim, d->l0_split, &P.net[0]))) return rc;
  P.n_obs = 1;
  P.n_per_obs = d->n;
  P.tiles_per_obs = static_cast<int>((d->n + kTileM - 1) / kTileM);
  P.n_tiles = P.tiles_per_obs;
  P.S = 1;
  P.T = 1.f;
  P.out = d->out;
  P.fx = d->x;
  P.fcond = d->cond;
  P.ft = d->t;
  P.fx_dim = d->x_dim;
  P.fcond_dim = d->cond_dim;
  P.out_dim = d->net.out_dim;
  return launch(P, s);
}

}  // namespace dmip
